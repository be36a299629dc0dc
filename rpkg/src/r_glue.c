/*
 * r_glue.c — `.Call` glue between the EasyLP R package and libeasylp_b200.so (include/easylp_abi.h).
 *
 * This is the file a maintainer of benet1one/EasyLP adds under src/ (with `useDynLib(easylp, .registration = TRUE)`
 * in NAMESPACE and `PKG_LIBS = -leasylp_b200` in src/Makevars).  It replaces the lpSolveAPI calls of `$solve()`
 * (/root/reference/R/class.R:260-278) with ONE `.Call`, and gives `$con()`/`$min()`/`$max()` a device assembly and
 * `private$feasible()` (R/class.R:533-540) a device re-check.  It is deliberately dumb: argument unpacking, index base
 * conversion (R is 1-based, the ABI 0-based), result lists.  No arithmetic happens here.
 *
 * R is not installed in the build image, so this file is only compiled against a minimal mock of R's C API
 * (tests/r_mock/) to keep it honest; it has never been executed.
 *
 * Conventions: inputs are read-only views of R vectors valid during the call; outputs are freshly allocated,
 * PROTECTed vectors; a nonzero return code of the library becomes an R error AFTER temporary memory is released
 * (R_alloc memory is reclaimed by R itself).
 */
#include <R.h>
#include <Rinternals.h>
#include <R_ext/Rdynload.h>
#include <stdint.h>
#include <string.h>

#include "easylp_abi.h"

static void elp_fail(const char* where) {
    char buf[1024];
    buf[0] = 0;
    elp_last_error(buf, (int32_t)sizeof buf);
    Rf_error("%s: %s", where, buf[0] ? buf : "unknown error in libeasylp_b200");
}

static SEXP named_list(int n, const char** names) {
    SEXP out = PROTECT(Rf_allocVector(VECSXP, n));
    SEXP nm = PROTECT(Rf_allocVector(STRSXP, n));
    for (int i = 0; i < n; ++i) SET_STRING_ELT(nm, i, Rf_mkChar(names[i]));
    Rf_setAttrib(out, R_NamesSymbol, nm);
    UNPROTECT(2);
    return out;
}

/* R `dir` strings -> sense codes.  strict != 0 keeps "<"/">" distinct (3/4) for check_feasible
 * (R/utils.R:167-171 uses match.fun(dir)); for the solver they fold onto "<="/">=" like lpSolveAPI does. */
static int8_t* sense_codes(SEXP dir, int strict) {
    const R_xlen_t m = XLENGTH(dir);
    int8_t* s = (int8_t*)R_alloc((size_t)(m > 0 ? m : 1), 1);
    for (R_xlen_t i = 0; i < m; ++i) {
        const char* d = CHAR(STRING_ELT(dir, i));
        if (!strcmp(d, "<=")) s[i] = ELP_LE;
        else if (!strcmp(d, ">=")) s[i] = ELP_GE;
        else if (!strcmp(d, "==") || !strcmp(d, "=")) s[i] = ELP_EQ;
        else if (!strcmp(d, "<")) s[i] = strict ? 3 : ELP_LE;
        else if (!strcmp(d, ">")) s[i] = strict ? 4 : ELP_GE;
        else Rf_error("unknown constraint direction '%s'", d);
    }
    return s;
}

static int32_t* zero_based(SEXP idx) {
    const R_xlen_t k = XLENGTH(idx);
    int32_t* out = (int32_t*)R_alloc((size_t)(k > 0 ? k : 1), sizeof(int32_t));
    const int* p = INTEGER(idx);
    for (R_xlen_t i = 0; i < k; ++i) out[i] = (int32_t)p[i] - 1;
    return out;
}

/* .Call("easylp_assemble_csr", term_row, term_col, term_val, m, n)
 * term_row / term_col: 1-based integer vectors in emission (fold) order.  Returns list(row_ptr, col_idx, vals)
 * with 0-based row_ptr and 1-based col_idx (ready for R indexing). */
SEXP easylp_assemble_csr(SEXP term_row, SEXP term_col, SEXP term_val, SEXP m_, SEXP n_) {
    const int64_t T = (int64_t)XLENGTH(term_val);
    const int32_t m = Rf_asInteger(m_), n = Rf_asInteger(n_);
    if (XLENGTH(term_row) != T || XLENGTH(term_col) != T) Rf_error("term vectors differ in length");
    int32_t* row = zero_based(term_row);
    int32_t* col = zero_based(term_col);
    int32_t* col_out = (int32_t*)R_alloc((size_t)(T > 0 ? T : 1), sizeof(int32_t));
    double* val_out = (double*)R_alloc((size_t)(T > 0 ? T : 1), sizeof(double));
    SEXP row_ptr = PROTECT(Rf_allocVector(INTSXP, (R_xlen_t)m + 1));
    int64_t nnz = 0;
    const int rc = elp_assemble_csr(T, row, col, REAL(term_val), m, n, (int32_t*)INTEGER(row_ptr), col_out, val_out, &nnz, NULL);
    if (rc) { UNPROTECT(1); elp_fail("easylp_assemble_csr"); }
    SEXP col_idx = PROTECT(Rf_allocVector(INTSXP, (R_xlen_t)nnz));
    SEXP vals = PROTECT(Rf_allocVector(REALSXP, (R_xlen_t)nnz));
    for (int64_t i = 0; i < nnz; ++i) INTEGER(col_idx)[i] = col_out[i] + 1;
    if (nnz) memcpy(REAL(vals), val_out, (size_t)nnz * sizeof(double));
    const char* names[] = {"row_ptr", "col_idx", "vals"};
    SEXP out = PROTECT(named_list(3, names));
    SET_VECTOR_ELT(out, 0, row_ptr);
    SET_VECTOR_ELT(out, 1, col_idx);
    SET_VECTOR_ELT(out, 2, vals);
    UNPROTECT(4);
    return out;
}

/* list(status, objval, x, y, stats) of a solve; x and y are PROTECTed by the caller */
static SEXP solve_result(int32_t status, double objval, SEXP x, SEXP y, const elp_stats* st) {
    const char* snames[] = {"method", "iterations", "restarts", "rel_primal_res", "rel_dual_res", "rel_gap",
                            "setup_ms", "solve_ms", "kernel_launches", "h2d_bytes", "d2h_bytes", "simplex_ctas"};
    SEXP stats = PROTECT(named_list(12, snames));
    SET_VECTOR_ELT(stats, 0, Rf_ScalarInteger(st->method_used));
    SET_VECTOR_ELT(stats, 1, Rf_ScalarInteger(st->iterations));
    SET_VECTOR_ELT(stats, 2, Rf_ScalarInteger(st->restarts));
    SET_VECTOR_ELT(stats, 3, Rf_ScalarReal(st->rel_primal_res));
    SET_VECTOR_ELT(stats, 4, Rf_ScalarReal(st->rel_dual_res));
    SET_VECTOR_ELT(stats, 5, Rf_ScalarReal(st->rel_gap));
    SET_VECTOR_ELT(stats, 6, Rf_ScalarReal(st->setup_ms));
    SET_VECTOR_ELT(stats, 7, Rf_ScalarReal(st->solve_ms));
    SET_VECTOR_ELT(stats, 8, Rf_ScalarReal((double)st->kernel_launches));
    SET_VECTOR_ELT(stats, 9, Rf_ScalarReal((double)st->h2d_bytes));
    SET_VECTOR_ELT(stats, 10, Rf_ScalarReal((double)st->d2h_bytes));
    SET_VECTOR_ELT(stats, 11, Rf_ScalarInteger(st->simplex_ctas));
    const char* names[] = {"status", "objval", "x", "y", "stats"};
    SEXP out = PROTECT(named_list(5, names));
    SET_VECTOR_ELT(out, 0, Rf_ScalarInteger(status));
    SET_VECTOR_ELT(out, 1, Rf_ScalarReal(objval));
    SET_VECTOR_ELT(out, 2, x);
    SET_VECTOR_ELT(out, 3, y);
    SET_VECTOR_ELT(out, 4, stats);
    UNPROTECT(2);
    return out;
}

static void fill_options(elp_options* opt, SEXP control) {
    /* `control`: named list built by `$solve(...)` from the arguments it used to forward to lp.control()
     * (R/class.R:262): timeout, epsilon, verbose are mapped; gpu.* are additive. */
    elp_default_options(opt);
    if (control == R_NilValue) return;
    SEXP nm = Rf_getAttrib(control, R_NamesSymbol);
    for (R_xlen_t i = 0; i < XLENGTH(control); ++i) {
        const char* k = CHAR(STRING_ELT(nm, i));
        SEXP v = VECTOR_ELT(control, i);
        if (!strcmp(k, "timeout")) opt->time_limit_s = Rf_asReal(v);
        /* lp_solve's `epsilon` is its INTEGER-ROUNDING tolerance (1e-9 / 1e-11 are usual values), not an optimality
         * tolerance: mapping it to PDLP's relative KKT tolerance drove solves to the iteration cap (ADVICE r1).  Only
         * gpu.tol sets eps_rel; `$solve()` warns that `epsilon` is ignored. */
        else if (!strcmp(k, "gpu.tol")) opt->eps_rel = Rf_asReal(v);
        else if (!strcmp(k, "gpu.devices")) opt->devices = Rf_asInteger(v);       /* GPUs of the box to spread one solve over */
        else if (!strcmp(k, "verbose")) opt->verbose = Rf_asInteger(v);
        else if (!strcmp(k, "gpu.max_iter")) opt->max_iter = Rf_asInteger(v);
        else if (!strcmp(k, "gpu.method")) opt->method = Rf_asInteger(v);
        else if (!strcmp(k, "gpu.transpose")) opt->transpose = Rf_asInteger(v);   /* 1: bit-reproducible CSC gather */
        /* everything else has no meaning on the GPU path; `$solve()` warns about it on the R side */
    }
}

/* .Call("easylp_solve_lp", row_ptr, col_idx, vals, dir, rhs, objective_fun, maximize, lower, upper, control)
 * Replaces make.lp/set.objfn/lp.control/set.bounds/add.constraint/solve/get.objective/get.variables
 * (R/class.R:260-278).  Returns list(status = <lp_solve code>, objval, x, y, stats). */
SEXP easylp_solve_lp(SEXP row_ptr, SEXP col_idx, SEXP vals, SEXP dir, SEXP rhs, SEXP cost, SEXP maximize,
                     SEXP lower, SEXP upper, SEXP control) {
    const int32_t m = (int32_t)XLENGTH(row_ptr) - 1, n = (int32_t)XLENGTH(cost);
    if (XLENGTH(lower) != n || XLENGTH(upper) != n) Rf_error("bounds must have one entry per variable");
    if (XLENGTH(dir) != m || XLENGTH(rhs) != m) Rf_error("dir/rhs must have one entry per constraint");
    elp_options opt;
    fill_options(&opt, control);
    int8_t* sense = sense_codes(dir, 0);
    int32_t* cols = zero_based(col_idx);
    SEXP x = PROTECT(Rf_allocVector(REALSXP, n));
    SEXP y = PROTECT(Rf_allocVector(REALSXP, m));
    int32_t status = 0;
    double objval = 0.0;
    elp_stats st;
    memset(&st, 0, sizeof st);
    const int rc = elp_solve_lp(m, n, (const int32_t*)INTEGER(row_ptr), cols, REAL(vals), sense, REAL(rhs), REAL(cost),
                                Rf_asLogical(maximize) ? 1 : 0, REAL(lower), REAL(upper), &opt, &status, &objval,
                                REAL(x), m > 0 ? REAL(y) : NULL, &st);
    if (rc) { UNPROTECT(2); elp_fail("easylp_solve_lp"); }
    SEXP out = solve_result(status, objval, x, y, &st);
    UNPROTECT(2);
    return out;
}

/* .Call("easylp_solve_mip", row_ptr, col_idx, vals, dir, rhs, objective_fun, maximize, lower, upper, is_integer, control)
 * Models with integer / binary variables: replaces set.type(prob, columns, type) + lp_solve's branch and bound behind
 * solve(prob) (R/class.R:264-276).  is_integer: logical(n), TRUE for integer and binary columns (binary columns carry the
 * bounds [0, 1], R/class.R:104-110).  Same result list as easylp_solve_lp (y is all zero: no duals for a MILP). */
SEXP easylp_solve_mip(SEXP row_ptr, SEXP col_idx, SEXP vals, SEXP dir, SEXP rhs, SEXP cost, SEXP maximize,
                      SEXP lower, SEXP upper, SEXP is_integer, SEXP control) {
    const int32_t m = (int32_t)XLENGTH(row_ptr) - 1, n = (int32_t)XLENGTH(cost);
    if (XLENGTH(lower) != n || XLENGTH(upper) != n || XLENGTH(is_integer) != n)
        Rf_error("bounds and types must have one entry per variable");
    if (XLENGTH(dir) != m || XLENGTH(rhs) != m) Rf_error("dir/rhs must have one entry per constraint");
    elp_options opt;
    fill_options(&opt, control);
    int8_t* sense = sense_codes(dir, 0);
    int32_t* cols = zero_based(col_idx);
    uint8_t* ii = (uint8_t*)R_alloc((size_t)(n > 0 ? n : 1), 1);
    for (int32_t j = 0; j < n; ++j) ii[j] = LOGICAL(is_integer)[j] ? 1 : 0;
    SEXP x = PROTECT(Rf_allocVector(REALSXP, n));
    SEXP y = PROTECT(Rf_allocVector(REALSXP, m));
    for (int32_t i = 0; i < m; ++i) REAL(y)[i] = 0.0;
    int32_t status = 0;
    double objval = 0.0;
    elp_stats st;
    memset(&st, 0, sizeof st);
    const int rc = elp_solve_mip(m, n, (const int32_t*)INTEGER(row_ptr), cols, REAL(vals), sense, REAL(rhs), REAL(cost),
                                 Rf_asLogical(maximize) ? 1 : 0, REAL(lower), REAL(upper), ii, &opt, &status, &objval,
                                 REAL(x), &st);
    if (rc) { UNPROTECT(2); elp_fail("easylp_solve_mip"); }
    SEXP out = solve_result(status, objval, x, y, &st);
    UNPROTECT(2);
    return out;
}

/* .Call("easylp_sensitivity", row_ptr, col_idx, vals, dir, rhs, objective_fun, maximize, lower, upper, control)
 * Replaces get.sensitivity.obj(prob) / get.sensitivity.rhs(prob) behind `$sensitivity_objective` / `$sensitivity_rhs`
 * (R/class.R:613-646).  Returns list(status, objfrom, objtill, rhsfrom, rhstill, duals); infinite ends are +/-Inf. */
SEXP easylp_sensitivity(SEXP row_ptr, SEXP col_idx, SEXP vals, SEXP dir, SEXP rhs, SEXP cost, SEXP maximize,
                        SEXP lower, SEXP upper, SEXP control) {
    const int32_t m = (int32_t)XLENGTH(row_ptr) - 1, n = (int32_t)XLENGTH(cost);
    if (XLENGTH(lower) != n || XLENGTH(upper) != n) Rf_error("bounds must have one entry per variable");
    if (XLENGTH(dir) != m || XLENGTH(rhs) != m) Rf_error("dir/rhs must have one entry per constraint");
    elp_options opt;
    fill_options(&opt, control);
    int8_t* sense = sense_codes(dir, 0);
    int32_t* cols = zero_based(col_idx);
    double* x = (double*)R_alloc((size_t)(n > 0 ? n : 1), sizeof(double));
    const char* names[] = {"status", "objfrom", "objtill", "rhsfrom", "rhstill", "duals"};
    SEXP out = PROTECT(named_list(6, names));
    SEXP of = PROTECT(Rf_allocVector(REALSXP, n)), ot = PROTECT(Rf_allocVector(REALSXP, n));
    SEXP rf = PROTECT(Rf_allocVector(REALSXP, m)), rt = PROTECT(Rf_allocVector(REALSXP, m)), du = PROTECT(Rf_allocVector(REALSXP, m));
    int32_t status = 0;
    double objval = 0.0;
    const int rc = elp_sensitivity(m, n, (const int32_t*)INTEGER(row_ptr), cols, REAL(vals), sense, REAL(rhs), REAL(cost),
                                   Rf_asLogical(maximize) ? 1 : 0, REAL(lower), REAL(upper), &opt, &status, &objval, x,
                                   REAL(of), REAL(ot), m > 0 ? REAL(rf) : NULL, m > 0 ? REAL(rt) : NULL, m > 0 ? REAL(du) : NULL);
    if (rc) { UNPROTECT(6); elp_fail("easylp_sensitivity"); }
    SET_VECTOR_ELT(out, 0, Rf_ScalarInteger(status));
    SET_VECTOR_ELT(out, 1, of); SET_VECTOR_ELT(out, 2, ot); SET_VECTOR_ELT(out, 3, rf); SET_VECTOR_ELT(out, 4, rt);
    SET_VECTOR_ELT(out, 5, du);
    UNPROTECT(6);
    return out;
}

/* .Call("easylp_check_feasible", row_ptr, col_idx, vals, sol, dir, rhs, tol) -> logical(m)
 * Replaces `lhs <- mat %*% sol` + compare_tol (R/class.R:533-540, R/utils.R:167-171). */
SEXP easylp_check_feasible(SEXP row_ptr, SEXP col_idx, SEXP vals, SEXP sol, SEXP dir, SEXP rhs, SEXP tol) {
    const int32_t m = (int32_t)XLENGTH(row_ptr) - 1, n = (int32_t)XLENGTH(sol);
    int8_t* sense = sense_codes(dir, 1);
    int32_t* cols = zero_based(col_idx);
    uint8_t* ok = (uint8_t*)R_alloc((size_t)(m > 0 ? m : 1), 1);
    const int rc = elp_check_feasible(m, n, (const int32_t*)INTEGER(row_ptr), cols, REAL(vals), REAL(sol), sense, REAL(rhs),
                                      Rf_asReal(tol), ok);
    if (rc) elp_fail("easylp_check_feasible");
    SEXP out = PROTECT(Rf_allocVector(LGLSXP, m));
    for (int32_t i = 0; i < m; ++i) LOGICAL(out)[i] = ok[i] ? 1 : 0;
    UNPROTECT(1);
    return out;
}

/* .Call("easylp_solve_batch", A, b, c, lower, upper, dir, maximize, control)
 * Additive entry point for BASELINE config 3: A is an array with dim c(n, m, B) (so that each LP's rows are
 * contiguous: R is column-major, the ABI wants [B][m][n] row-major), b is m x B, c/lower/upper are n x B,
 * dir a character vector of length m (recycled over the batch) or NULL for all "<=".
 * Returns list(status = integer(B), objval = numeric(B), x = matrix(n, B)). */
SEXP easylp_solve_batch(SEXP A, SEXP b, SEXP c, SEXP lower, SEXP upper, SEXP dir, SEXP maximize, SEXP control) {
    SEXP dim = Rf_getAttrib(A, R_DimSymbol);
    if (dim == R_NilValue || XLENGTH(dim) != 3) Rf_error("A must be an n x m x B array");
    const int32_t n = INTEGER(dim)[0], m = INTEGER(dim)[1];
    const int64_t B = INTEGER(dim)[2];
    elp_options opt;
    fill_options(&opt, control);
    int8_t* sense = NULL;
    if (dir != R_NilValue) {
        if (XLENGTH(dir) != m) Rf_error("dir must have one entry per constraint");
        int8_t* one = sense_codes(dir, 0);
        sense = (int8_t*)R_alloc((size_t)(B * m > 0 ? B * m : 1), 1);
        for (int64_t k = 0; k < B; ++k) memcpy(sense + k * m, one, (size_t)m);
    }
    SEXP status = PROTECT(Rf_allocVector(INTSXP, (R_xlen_t)B));
    SEXP obj = PROTECT(Rf_allocVector(REALSXP, (R_xlen_t)B));
    SEXP x = PROTECT(Rf_allocMatrix(REALSXP, n, (int)B));
    const int rc = elp_solve_batch(B, m, n, REAL(A), REAL(b), REAL(c), lower == R_NilValue ? NULL : REAL(lower),
                                   upper == R_NilValue ? NULL : REAL(upper), sense, Rf_asLogical(maximize) ? 1 : 0, &opt,
                                   (int32_t*)INTEGER(status), REAL(obj), REAL(x), NULL);
    if (rc) { UNPROTECT(3); elp_fail("easylp_solve_batch"); }
    const char* names[] = {"status", "objval", "x"};
    SEXP out = PROTECT(named_list(3, names));
    SET_VECTOR_ELT(out, 0, status);
    SET_VECTOR_ELT(out, 1, obj);
    SET_VECTOR_ELT(out, 2, x);
    UNPROTECT(4);
    return out;
}

/* Element `name` of a named R list, or R_NilValue. */
static SEXP list_get(SEXP lst, const char* name) {
    SEXP nm = Rf_getAttrib(lst, R_NamesSymbol);
    if (nm == R_NilValue) return R_NilValue;
    for (R_xlen_t i = 0; i < XLENGTH(lst); ++i)
        if (!strcmp(CHAR(STRING_ELT(nm, i)), name)) return VECTOR_ELT(lst, i);
    return R_NilValue;
}

/* .Call("easylp_assemble_lowered", term_row, term_col, term_val, families, groups, m, n)
 * The lowered assembly (include/easylp_abi.h, "(1b)"): `for (v in seq) body` / `sum_for(i = I, body)` whose body the R
 * side recognised with substitute() as affine in indexed variables arrive as FAMILIES instead of expanded terms.
 *   families: list of lists with integer scalars `out_offset`, `out_stride`, `group` (1-based), `row0` (1-based),
 *             `col0` (1-based), integer vectors `extent`, `row_stride`, `coef_stride` (one entry per loop, slowest first),
 *             lists `col_tab` / `row_tab` (per loop an integer vector of 0-based offsets, or NULL) and a double vector
 *             `coef`.
 *   groups:   list of lists with `row0` (1-based) and `mul`, a list of double vectors (length 1 = scalar, else one
 *             multiplier per row of the block); group 1 is the plain group of the explicit terms.
 * Returns list(row_ptr, col_idx, vals) like easylp_assemble_csr. */
typedef struct {
    elp_term_family* fam;
    elp_fold_group* grp;
    int32_t* itab;
    double* dtab;
    int32_t nf, ng;
    int64_t ni, nd, total;
} packed_families;

/* R lists of families / groups -> the ABI's structs and pooled tables (R_alloc memory: reclaimed by R) */
static packed_families pack_families(SEXP families, SEXP groups) {
    packed_families P;
    P.nf = (int32_t)XLENGTH(families);
    P.ng = (int32_t)XLENGTH(groups);
    P.ni = P.nd = P.total = 0;
    for (int32_t f = 0; f < P.nf; ++f) {           /* pass 1: table sizes */
        SEXP F = VECTOR_ELT(families, f);
        SEXP ext = list_get(F, "extent"), ct = list_get(F, "col_tab"), rt = list_get(F, "row_tab");
        const R_xlen_t nl = XLENGTH(ext);
        if (nl > ELP_MAX_LOOPS) Rf_error("family %d has %d loops (max %d)", f + 1, (int)nl, ELP_MAX_LOOPS);
        int64_t cnt = 1;
        for (R_xlen_t l = 0; l < nl; ++l) {
            cnt *= INTEGER(ext)[l];
            if (ct != R_NilValue && VECTOR_ELT(ct, l) != R_NilValue) P.ni += XLENGTH(VECTOR_ELT(ct, l));
            if (rt != R_NilValue && VECTOR_ELT(rt, l) != R_NilValue) P.ni += XLENGTH(VECTOR_ELT(rt, l));
        }
        P.nd += XLENGTH(list_get(F, "coef"));
        P.total += cnt;
    }
    for (int32_t g = 0; g < P.ng; ++g) {
        SEXP mul = list_get(VECTOR_ELT(groups, g), "mul");
        if (mul != R_NilValue) for (R_xlen_t k = 0; k < XLENGTH(mul); ++k) P.nd += XLENGTH(VECTOR_ELT(mul, k));
    }
    P.fam = (elp_term_family*)R_alloc((size_t)(P.nf > 0 ? P.nf : 1), sizeof(elp_term_family));
    P.grp = (elp_fold_group*)R_alloc((size_t)(P.ng > 0 ? P.ng : 1), sizeof(elp_fold_group));
    P.itab = (int32_t*)R_alloc((size_t)(P.ni > 0 ? P.ni : 1), sizeof(int32_t));
    P.dtab = (double*)R_alloc((size_t)(P.nd > 0 ? P.nd : 1), sizeof(double));
    int64_t pi = 0, pd = 0;                        /* pass 2: pack */
    for (int32_t g = 0; g < P.ng; ++g) {
        SEXP G = VECTOR_ELT(groups, g), mul = list_get(G, "mul");
        memset(&P.grp[g], 0, sizeof P.grp[g]);
        P.grp[g].row0 = Rf_asInteger(list_get(G, "row0")) - 1;
        P.grp[g].n_mul = mul == R_NilValue ? 0 : (int32_t)XLENGTH(mul);
        if (P.grp[g].n_mul > ELP_MAX_GROUP_MUL) Rf_error("group %d has too many multipliers", g + 1);
        for (int32_t k = 0; k < P.grp[g].n_mul; ++k) {
            SEXP v = VECTOR_ELT(mul, k);
            P.grp[g].mul_tab[k] = pd;
            P.grp[g].mul_per_row[k] = XLENGTH(v) > 1;
            memcpy(P.dtab + pd, REAL(v), (size_t)XLENGTH(v) * sizeof(double));
            pd += XLENGTH(v);
        }
    }
    for (int32_t f = 0; f < P.nf; ++f) {
        SEXP F = VECTOR_ELT(families, f);
        SEXP ext = list_get(F, "extent"), rs = list_get(F, "row_stride"), cs = list_get(F, "coef_stride");
        SEXP ct = list_get(F, "col_tab"), rt = list_get(F, "row_tab"), coef = list_get(F, "coef");
        elp_term_family* t = &P.fam[f];
        memset(t, 0, sizeof *t);
        t->n_loops = (int32_t)XLENGTH(ext);
        t->out_offset = (int64_t)Rf_asReal(list_get(F, "out_offset"));
        t->out_stride = Rf_asInteger(list_get(F, "out_stride"));
        t->group = Rf_asInteger(list_get(F, "group")) - 1;
        t->row0 = Rf_asInteger(list_get(F, "row0")) - 1;
        t->col0 = Rf_asInteger(list_get(F, "col0")) - 1;
        t->coef_tab = pd;
        memcpy(P.dtab + pd, REAL(coef), (size_t)XLENGTH(coef) * sizeof(double));
        pd += XLENGTH(coef);
        t->count = 1;
        for (int32_t l = 0; l < t->n_loops; ++l) {
            t->extent[l] = INTEGER(ext)[l];
            t->row_stride[l] = INTEGER(rs)[l];
            t->coef_stride[l] = INTEGER(cs)[l];
            t->count *= t->extent[l];
            t->col_tab[l] = t->row_tab[l] = -1;
            SEXP c = ct == R_NilValue ? R_NilValue : VECTOR_ELT(ct, l);
            SEXP r = rt == R_NilValue ? R_NilValue : VECTOR_ELT(rt, l);
            if (c != R_NilValue) { t->col_tab[l] = pi; memcpy(P.itab + pi, INTEGER(c), (size_t)XLENGTH(c) * sizeof(int32_t)); pi += XLENGTH(c); }
            if (r != R_NilValue) { t->row_tab[l] = pi; memcpy(P.itab + pi, INTEGER(r), (size_t)XLENGTH(r) * sizeof(int32_t)); pi += XLENGTH(r); }
        }
    }
    return P;
}

static SEXP csr_list(SEXP row_ptr, const int32_t* col_out, const double* val_out, int64_t nnz) {
    SEXP col_idx = PROTECT(Rf_allocVector(INTSXP, (R_xlen_t)nnz));
    SEXP vals = PROTECT(Rf_allocVector(REALSXP, (R_xlen_t)nnz));
    for (int64_t i = 0; i < nnz; ++i) INTEGER(col_idx)[i] = col_out[i] + 1;
    if (nnz) memcpy(REAL(vals), val_out, (size_t)nnz * sizeof(double));
    const char* names[] = {"row_ptr", "col_idx", "vals"};
    SEXP out = PROTECT(named_list(3, names));
    SET_VECTOR_ELT(out, 0, row_ptr);
    SET_VECTOR_ELT(out, 1, col_idx);
    SET_VECTOR_ELT(out, 2, vals);
    UNPROTECT(3);
    return out;
}

SEXP easylp_assemble_lowered(SEXP term_row, SEXP term_col, SEXP term_val, SEXP families, SEXP groups, SEXP m_, SEXP n_) {
    const int64_t T = (int64_t)XLENGTH(term_val);
    const int32_t m = Rf_asInteger(m_), n = Rf_asInteger(n_);
    if (XLENGTH(term_row) != T || XLENGTH(term_col) != T) Rf_error("term vectors differ in length");
    const packed_families P = pack_families(families, groups);
    const int64_t cap = T + P.total > 0 ? T + P.total : 1;
    int32_t* row = zero_based(term_row);
    int32_t* col = zero_based(term_col);
    int32_t* col_out = (int32_t*)R_alloc((size_t)cap, sizeof(int32_t));
    double* val_out = (double*)R_alloc((size_t)cap, sizeof(double));
    SEXP row_ptr = PROTECT(Rf_allocVector(INTSXP, (R_xlen_t)m + 1));
    int64_t nnz = 0;
    const int rc = elp_assemble_lowered(T, row, col, REAL(term_val), P.nf, P.fam, P.ni, P.itab, P.nd, P.dtab, P.ng, P.grp, m, n,
                                        (int32_t*)INTEGER(row_ptr), col_out, val_out, cap, &nnz, NULL);
    if (rc) { UNPROTECT(1); elp_fail("easylp_assemble_lowered"); }
    SEXP out = csr_list(row_ptr, col_out, val_out, nnz);
    UNPROTECT(1);
    return out;
}

/* ---- device-resident model (include/easylp_abi.h "(1c)"): an external pointer whose finalizer frees the HBM copy.
 * The R object treats it as a rebuildable cache: `$clone()` and saveRDS() drop it, the next `$solve()` re-assembles. ---- */
static void model_finalizer(SEXP ptr) {
    elp_model* h = (elp_model*)R_ExternalPtrAddr(ptr);
    if (h) { elp_model_destroy(h); R_ClearExternalPtr(ptr); }
}

static elp_model* model_of(SEXP ptr) {
    elp_model* h = (elp_model*)R_ExternalPtrAddr(ptr);
    if (!h) Rf_error("the device copy of this model is gone (cloned or restored object): call $con()/$solve() again");
    return h;
}

/* .Call("easylp_model_assemble", term_row, term_col, term_val, families, groups, m, n) -> external pointer */
SEXP easylp_model_assemble(SEXP term_row, SEXP term_col, SEXP term_val, SEXP families, SEXP groups, SEXP m_, SEXP n_) {
    const int64_t T = (int64_t)XLENGTH(term_val);
    const int32_t m = Rf_asInteger(m_), n = Rf_asInteger(n_);
    if (XLENGTH(term_row) != T || XLENGTH(term_col) != T) Rf_error("term vectors differ in length");
    const packed_families P = pack_families(families, groups);
    elp_model* h = NULL;
    const int rc = elp_model_assemble(T, zero_based(term_row), zero_based(term_col), REAL(term_val), P.nf, P.fam, P.ni, P.itab,
                                      P.nd, P.dtab, P.ng, P.grp, m, n, &h, NULL, NULL);
    if (rc) elp_fail("easylp_model_assemble");
    SEXP ptr = PROTECT(R_MakeExternalPtr(h, R_NilValue, R_NilValue));
    R_RegisterCFinalizerEx(ptr, model_finalizer, TRUE);
    UNPROTECT(1);
    return ptr;
}

/* .Call("easylp_model_csr", model) -> list(row_ptr, col_idx, vals): `constraint$mat` for printing / inspection */
SEXP easylp_model_csr(SEXP model) {
    elp_model* h = model_of(model);
    int32_t m = 0, n = 0;
    int64_t nnz = 0;
    if (elp_model_dims(h, &m, &n, &nnz)) elp_fail("easylp_model_csr");
    int32_t* col_out = (int32_t*)R_alloc((size_t)(nnz > 0 ? nnz : 1), sizeof(int32_t));
    double* val_out = (double*)R_alloc((size_t)(nnz > 0 ? nnz : 1), sizeof(double));
    SEXP row_ptr = PROTECT(Rf_allocVector(INTSXP, (R_xlen_t)m + 1));
    if (elp_model_csr(h, (int32_t*)INTEGER(row_ptr), col_out, val_out)) { UNPROTECT(1); elp_fail("easylp_model_csr"); }
    SEXP out = csr_list(row_ptr, col_out, val_out, nnz);
    UNPROTECT(1);
    return out;
}

static void check_interrupt(void* unused) { (void)unused; R_CheckUserInterrupt(); }

/* .Call("easylp_model_solve", model, dir, rhs, objective_fun, maximize, lower, upper, control): `$solve()` on the
 * device-resident matrix; same result list as easylp_solve_lp. */
SEXP easylp_model_solve(SEXP model, SEXP dir, SEXP rhs, SEXP cost, SEXP maximize, SEXP lower, SEXP upper, SEXP control) {
    elp_model* h = model_of(model);
    int32_t m = 0, n = 0;
    if (elp_model_dims(h, &m, &n, NULL)) elp_fail("easylp_model_solve");
    if (XLENGTH(cost) != n || XLENGTH(lower) != n || XLENGTH(upper) != n) Rf_error("objective/bounds must have one entry per variable");
    if (XLENGTH(dir) != m || XLENGTH(rhs) != m) Rf_error("dir/rhs must have one entry per constraint");
    elp_options opt;
    fill_options(&opt, control);
    int8_t* sense = sense_codes(dir, 0);
    SEXP x = PROTECT(Rf_allocVector(REALSXP, n));
    SEXP y = PROTECT(Rf_allocVector(REALSXP, m));
    int32_t status = 0;
    double objval = 0.0;
    elp_stats st;
    memset(&st, 0, sizeof st);
    int rc;
    for (R_xlen_t j = 0; j < n; ++j)       /* lower > upper: "unfeasible" without a solve (R/class.R:297-298), as solve_large does */
        if (REAL(lower)[j] > REAL(upper)[j]) { opt.method = ELP_METHOD_AUTO; break; }
    if (opt.method == ELP_METHOD_PDLP && opt.devices <= 1) {
        /* a long first-order solve: run it in chunks and let the user interrupt between them (SURVEY 8b).
         * R_CheckUserInterrupt() would longjmp past our cleanup, so it runs under R_ToplevelExec. */
        elp_pdlp* p = NULL;
        rc = elp_model_pdlp_create(h, sense, REAL(rhs), REAL(cost), Rf_asLogical(maximize) ? 1 : 0, REAL(lower), REAL(upper),
                                   &opt, &p, &st);
        const double setup_ms = st.setup_ms;
        int interrupted = 0;
        int32_t seen = -1;
        while (!rc && !interrupted) {
            rc = elp_pdlp_run(p, 4096, &st);
            /* stop on an answer, on the solve's own iteration / time limit (the handle keeps the clock across calls and
             * says so in limit_reached), or when a call made no progress — never spin on a solve that cannot advance */
            if (rc || st.status != ELP_STATUS_TIMEOUT || st.limit_reached != 0 || st.iterations <= seen) break;
            seen = st.iterations;
            interrupted = !R_ToplevelExec(check_interrupt, NULL);
        }
        if (!rc && !interrupted) rc = elp_pdlp_solution(p, REAL(x), m > 0 ? REAL(y) : NULL, &objval);
        status = st.status;
        st.setup_ms = setup_ms;
        if (p) elp_pdlp_destroy(p);
        if (interrupted) { UNPROTECT(2); Rf_error("easylp$solve interrupted after %d PDHG iterations", st.iterations); }
        if (!rc && status == ELP_STATUS_UNBOUNDED) objval = Rf_asLogical(maximize) ? R_PosInf : R_NegInf;
    } else {
        rc = elp_model_solve(h, sense, REAL(rhs), REAL(cost), Rf_asLogical(maximize) ? 1 : 0, REAL(lower), REAL(upper),
                             &opt, &status, &objval, REAL(x), m > 0 ? REAL(y) : NULL, &st);
    }
    if (rc) { UNPROTECT(2); elp_fail("easylp_model_solve"); }
    SEXP out = solve_result(status, objval, x, y, &st);
    UNPROTECT(2);
    return out;
}

/* .Call("easylp_model_valid", model) -> TRUE when the external pointer still holds a device model (FALSE after a
 * clone / readRDS, whose pointers are NULL): `$solve()` rebuilds only then, and lets every real error propagate. */
SEXP easylp_model_valid(SEXP model) {
    return Rf_ScalarLogical(TYPEOF(model) == EXTPTRSXP && R_ExternalPtrAddr(model) != NULL);
}

/* .Call("easylp_device_count") */
SEXP easylp_device_count(void) {
    int32_t k = 0;
    if (elp_device_count(&k)) k = 0;
    return Rf_ScalarInteger(k);
}

static const R_CallMethodDef call_methods[] = {
    {"easylp_assemble_csr", (DL_FUNC)&easylp_assemble_csr, 5},
    {"easylp_assemble_lowered", (DL_FUNC)&easylp_assemble_lowered, 7},
    {"easylp_model_assemble", (DL_FUNC)&easylp_model_assemble, 7},
    {"easylp_model_csr", (DL_FUNC)&easylp_model_csr, 1},
    {"easylp_model_solve", (DL_FUNC)&easylp_model_solve, 8},
    {"easylp_model_valid", (DL_FUNC)&easylp_model_valid, 1},
    {"easylp_solve_lp", (DL_FUNC)&easylp_solve_lp, 10},
    {"easylp_solve_mip", (DL_FUNC)&easylp_solve_mip, 11},
    {"easylp_sensitivity", (DL_FUNC)&easylp_sensitivity, 10},
    {"easylp_check_feasible", (DL_FUNC)&easylp_check_feasible, 7},
    {"easylp_solve_batch", (DL_FUNC)&easylp_solve_batch, 8},
    {"easylp_device_count", (DL_FUNC)&easylp_device_count, 0},
    {NULL, NULL, 0}};

void R_init_easylp(DllInfo* dll) {
    R_registerRoutines(dll, NULL, call_methods, NULL, NULL);
    R_useDynamicSymbols(dll, FALSE);
}
