"""ctypes binding of libeasylp_b200.so (include/easylp_abi.h).

This is the Python twin of the R `.Call` glue in rpkg/src/r_glue.c: it only marshals plain buffers across
the C ABI.  There is NO CPU fallback — if the shared library is missing, or no CUDA device is present,
every compute call raises.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# ELP_LIB_PATH: another build of the same library (A/B runs of two kernel versions in one GPU call); default in-tree
LIB_PATH = os.environ.get("ELP_LIB_PATH") or os.path.join(_HERE, "libeasylp_b200.so")

LE, GE, EQ = 0, 1, 2
STATUS_OPTIMAL, STATUS_INFEASIBLE, STATUS_UNBOUNDED, STATUS_NUMFAILURE, STATUS_TIMEOUT = 0, 2, 3, 5, 7
METHOD_AUTO, METHOD_SIMPLEX, METHOD_PDLP = 0, 1, 2
TRANSPOSE_AUTO, TRANSPOSE_GATHER, TRANSPOSE_SCATTER = 0, 1, 2
UNIQUE_ID_BYTES = 128


class ElpError(RuntimeError):
    pass


class Options(C.Structure):
    _fields_ = [("eps_rel", C.c_double), ("time_limit_s", C.c_double), ("max_iter", C.c_int32),
                ("check_every", C.c_int32), ("method", C.c_int32), ("verbose", C.c_int32),
                ("use_graph", C.c_int32), ("ruiz_iters", C.c_int32), ("transpose", C.c_int32),
                ("devices", C.c_int32)]


class Stats(C.Structure):
    _fields_ = [("status", C.c_int32), ("method_used", C.c_int32), ("iterations", C.c_int32),
                ("restarts", C.c_int32), ("primal_obj", C.c_double), ("dual_obj", C.c_double),
                ("rel_primal_res", C.c_double), ("rel_dual_res", C.c_double), ("rel_gap", C.c_double),
                ("setup_ms", C.c_double), ("solve_ms", C.c_double), ("total_ms", C.c_double),
                ("kernel_launches", C.c_int64), ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64),
                ("spmv_ms", C.c_double), ("limit_reached", C.c_int32), ("simplex_ctas", C.c_int32)]

    def asdict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


# every symbol include/easylp_abi.h declares (tests/test_abi_symbols.py checks the header against this)
ABI_SYMBOLS = [
    "elp_version", "elp_last_error", "elp_device_count", "elp_set_device", "elp_default_options",
    "elp_status_string", "elp_kernel_launches", "elp_release_workspace", "elp_assemble_csr", "elp_assemble_lowered",
    "elp_expand_terms", "elp_model_assemble", "elp_model_dims", "elp_model_csr", "elp_model_solve", "elp_model_destroy", "elp_model_pdlp_create",
    "elp_solve_lp", "elp_solve_mip", "elp_sensitivity", "elp_solve_batch",
    "elp_batch_create", "elp_batch_run", "elp_batch_fetch", "elp_batch_destroy", "elp_spmv",
    "elp_check_feasible", "elp_pdlp_create", "elp_pdlp_run", "elp_pdlp_reset", "elp_pdlp_solution",
    "elp_pdlp_probe_spmv", "elp_pdlp_probe_step", "elp_pdlp_transpose", "elp_pdlp_destroy", "elp_comm_unique_id", "elp_comm_init", "elp_comm_size",
    "elp_comm_destroy",
]

_lib = None


def lib():
    """Loads the shared library (once).  Raises if it has not been built: no fallback exists."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ElpError(f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                           "or `make -C easylp_b200/csrc`.  There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        L.elp_version.restype = C.c_char_p
        L.elp_status_string.restype = C.c_char_p
        L.elp_status_string.argtypes = [C.c_int32]
        L.elp_kernel_launches.restype = C.c_int64
        _lib = L
    return _lib


def _check(rc):
    if rc != 0:
        buf = C.create_string_buffer(2048)
        lib().elp_last_error(buf, 2048)
        raise ElpError(buf.value.decode(errors="replace"))


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _f64(a, shape=None):
    if a is None:
        return None
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None and a.shape != tuple(shape):
        a = np.ascontiguousarray(np.broadcast_to(a, shape))
    return a


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def _i8(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.int8)


def version() -> str:
    return lib().elp_version().decode()


def device_count() -> int:
    c = C.c_int32(0)
    _check(lib().elp_device_count(C.byref(c)))
    return c.value


def set_device(dev: int):
    _check(lib().elp_set_device(C.c_int32(dev)))


def status_string(status: int) -> str:
    return lib().elp_status_string(C.c_int32(status)).decode()


def kernel_launches() -> int:
    return int(lib().elp_kernel_launches())


def release_workspace() -> None:
    """Frees the calling thread's cached device scratch (the assembly keeps a grow-only workspace)."""
    _check(lib().elp_release_workspace())


def default_options(**kw) -> Options:
    o = Options()
    _check(lib().elp_default_options(C.byref(o)))
    for k, v in kw.items():
        if not hasattr(o, k):
            raise TypeError(f"unknown option {k}")
        setattr(o, k, v)
    return o


def assemble_csr(term_row, term_col, term_val, m: int, n: int):
    """terms (emission order) -> canonical CSR (row_ptr, col_idx, vals), bit-exact left-fold of duplicates."""
    term_row, term_col = _i32(term_row), _i32(term_col)
    term_val = _f64(term_val)
    T = term_row.size
    assert term_col.size == T and term_val.size == T
    row_ptr = np.zeros(m + 1, np.int32)
    col_idx = np.zeros(max(T, 1), np.int32)
    vals = np.zeros(max(T, 1), np.float64)
    nnz = C.c_int64(0)
    st = Stats()
    _check(lib().elp_assemble_csr(C.c_int64(T), _p(term_row), _p(term_col), _p(term_val), C.c_int32(m), C.c_int32(n),
                                  _p(row_ptr), _p(col_idx), _p(vals), C.byref(nnz), C.byref(st)))
    k = nnz.value
    return row_ptr, col_idx[:k].copy(), vals[:k].copy(), st


def assemble_lowered(term_row, term_col, term_val, packed, m: int, n: int):
    """explicit terms + index-set families (lower.pack) -> canonical CSR; the families are expanded on the device."""
    fam, n_fam, itab, dtab, grp, n_grp, n_low = packed
    term_row, term_col = _i32(term_row), _i32(term_col)
    term_val = _f64(term_val)
    T = term_row.size
    cap = max(T + n_low, 1)
    row_ptr = np.zeros(m + 1, np.int32)
    col_idx = np.zeros(cap, np.int32)
    vals = np.zeros(cap, np.float64)
    nnz = C.c_int64(0)
    st = Stats()
    _check(lib().elp_assemble_lowered(C.c_int64(T), _p(term_row), _p(term_col), _p(term_val), C.c_int32(n_fam), fam,
                                      C.c_int64(itab.size), _p(itab), C.c_int64(dtab.size), _p(dtab), C.c_int32(n_grp), grp,
                                      C.c_int32(m), C.c_int32(n), _p(row_ptr), _p(col_idx), _p(vals), C.c_int64(cap),
                                      C.byref(nnz), C.byref(st)))
    k = nnz.value
    return row_ptr, col_idx[:k].copy(), vals[:k].copy(), st


class Model:
    """Device-resident canonical CSR of one model (elp_model_*): assembled from explicit terms and/or index-set families,
    solved without the matrix crossing PCIe again, copied back only when the host asks for it."""

    def __init__(self, term_row, term_col, term_val, packed, m: int, n: int):
        fam, n_fam, itab, dtab, grp, n_grp, _n_low = packed
        term_row, term_col = _i32(term_row), _i32(term_col)
        term_val = _f64(term_val)
        self.m, self.n = int(m), int(n)
        self._h = C.c_void_p()
        nnz = C.c_int64(0)
        self.stats = Stats()
        _check(lib().elp_model_assemble(C.c_int64(term_row.size), _p(term_row), _p(term_col), _p(term_val), C.c_int32(n_fam),
                                        fam, C.c_int64(itab.size), _p(itab), C.c_int64(dtab.size), _p(dtab),
                                        C.c_int32(n_grp), grp, C.c_int32(m), C.c_int32(n), C.byref(self._h),
                                        C.byref(nnz), C.byref(self.stats)))
        self.nnz = nnz.value

    def csr(self):
        row_ptr = np.zeros(self.m + 1, np.int32)
        col_idx = np.zeros(max(self.nnz, 1), np.int32)
        vals = np.zeros(max(self.nnz, 1), np.float64)
        _check(lib().elp_model_csr(self._h, _p(row_ptr), _p(col_idx), _p(vals)))
        return row_ptr, col_idx[:self.nnz], vals[:self.nnz]

    def solve(self, sense, rhs, c, lb, ub, maximize=False, options: Options | None = None):
        n, m = self.n, self.m
        rhs, c = _f64(rhs), _f64(c)
        lb, ub = _f64(lb, (n,)), _f64(ub, (n,))
        sense = _i8(sense)
        x = np.zeros(n)
        y = np.zeros(max(m, 1))
        status = C.c_int32(-1)
        obj = C.c_double(np.nan)
        st = Stats()
        _check(lib().elp_model_solve(self._h, _p(sense), _p(rhs), _p(c), C.c_int32(1 if maximize else 0), _p(lb), _p(ub),
                                     C.byref(options) if options is not None else None, C.byref(status), C.byref(obj),
                                     _p(x), _p(y), C.byref(st)))
        return LpResult(status.value, obj.value, x, y[:m], st)

    def pdlp(self, sense, rhs, c, lb, ub, maximize=False, options: Options | None = None) -> "Pdlp":
        """a PDLP handle on this device-resident matrix (run it in chunks with .run(k), as the R glue does)"""
        n = self.n
        rhs, c = _f64(rhs), _f64(c)
        lb, ub = _f64(lb, (n,)), _f64(ub, (n,))
        sense = _i8(sense)
        h = Pdlp.__new__(Pdlp)
        h.m, h.n = self.m, self.n
        h._h = C.c_void_p()
        h.setup_stats = Stats()
        h._keep = (sense, rhs, c, lb, ub)
        _check(lib().elp_model_pdlp_create(self._h, _p(sense), _p(rhs), _p(c), C.c_int32(1 if maximize else 0), _p(lb),
                                           _p(ub), C.byref(options) if options is not None else None, C.byref(h._h),
                                           C.byref(h.setup_stats)))
        return h

    def __deepcopy__(self, memo):         # a clone of the model rebuilds its own device copy (`$clone()`, SURVEY 8b)
        return None

    def close(self):
        if self._h:
            lib().elp_model_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def expand_terms(packed):
    """the term stream the device expands the families into: (row, col, val, group) — tests"""
    fam, n_fam, itab, dtab, _grp, _n_grp, n_low = packed
    row, col = np.zeros(max(n_low, 1), np.int32), np.zeros(max(n_low, 1), np.int32)
    val, grp = np.zeros(max(n_low, 1)), np.zeros(max(n_low, 1), np.int32)
    _check(lib().elp_expand_terms(C.c_int32(n_fam), fam, C.c_int64(itab.size), _p(itab), C.c_int64(dtab.size), _p(dtab),
                                  _p(row), _p(col), _p(val), _p(grp)))
    return row[:n_low], col[:n_low], val[:n_low], grp[:n_low]


@dataclass
class LpResult:
    status: int
    objval: float
    x: np.ndarray
    y: np.ndarray
    stats: Stats

    @property
    def status_string(self):
        return status_string(self.status)


def solve_lp(m, n, row_ptr, col_idx, vals, sense, rhs, c, lb, ub, maximize=False, options: Options | None = None):
    row_ptr, col_idx = _i32(row_ptr), _i32(col_idx)
    vals, rhs, c = _f64(vals), _f64(rhs), _f64(c)
    lb, ub = _f64(lb, (n,)), _f64(ub, (n,))
    sense = _i8(sense)
    if row_ptr.size == 0:
        row_ptr = np.zeros(1, np.int32)
    x = np.zeros(n)
    y = np.zeros(max(m, 1))
    status = C.c_int32(-1)
    obj = C.c_double(np.nan)
    st = Stats()
    _check(lib().elp_solve_lp(C.c_int32(m), C.c_int32(n), _p(row_ptr), _p(col_idx), _p(vals), _p(sense), _p(rhs), _p(c),
                              C.c_int32(1 if maximize else 0), _p(lb), _p(ub),
                              C.byref(options) if options is not None else None,
                              C.byref(status), C.byref(obj), _p(x), _p(y), C.byref(st)))
    return LpResult(status.value, obj.value, x, y[:m], st)


def solve_mip(m, n, row_ptr, col_idx, vals, sense, rhs, c, lb, ub, is_integer, maximize=False,
              options: Options | None = None):
    """branch and bound over the batched simplex kernel (elp_solve_mip); is_integer marks the integer columns"""
    row_ptr, col_idx = _i32(row_ptr), _i32(col_idx)
    vals, rhs, c = _f64(vals), _f64(rhs), _f64(c)
    lb, ub = _f64(lb, (n,)), _f64(ub, (n,))
    sense = _i8(sense)
    ii = np.ascontiguousarray(np.broadcast_to(is_integer, (n,)), dtype=np.uint8)
    if row_ptr.size == 0:
        row_ptr = np.zeros(1, np.int32)
    x = np.zeros(n)
    status = C.c_int32(-1)
    obj = C.c_double(np.nan)
    st = Stats()
    _check(lib().elp_solve_mip(C.c_int32(m), C.c_int32(n), _p(row_ptr), _p(col_idx), _p(vals), _p(sense), _p(rhs), _p(c),
                               C.c_int32(1 if maximize else 0), _p(lb), _p(ub), _p(ii),
                               C.byref(options) if options is not None else None,
                               C.byref(status), C.byref(obj), _p(x), C.byref(st)))
    return LpResult(status.value, obj.value, x, np.zeros(m), st)


def sensitivity(m, n, row_ptr, col_idx, vals, sense, rhs, c, lb, ub, maximize=False, options: Options | None = None):
    """elp_sensitivity: solve on the simplex path and range the objective coefficients and the right-hand sides.
    Returns (status, objval, x, obj_from, obj_till, rhs_from, rhs_till, duals)."""
    row_ptr, col_idx = _i32(row_ptr), _i32(col_idx)
    vals, rhs, c = _f64(vals), _f64(rhs), _f64(c)
    lb, ub = _f64(lb, (n,)), _f64(ub, (n,))
    sense = _i8(sense)
    if row_ptr.size == 0:
        row_ptr = np.zeros(1, np.int32)
    x, of, ot = np.zeros(n), np.zeros(n), np.zeros(n)
    rf, rt, du = np.zeros(max(m, 1)), np.zeros(max(m, 1)), np.zeros(max(m, 1))
    status = C.c_int32(-1)
    obj = C.c_double(np.nan)
    _check(lib().elp_sensitivity(C.c_int32(m), C.c_int32(n), _p(row_ptr), _p(col_idx), _p(vals), _p(sense), _p(rhs), _p(c),
                                 C.c_int32(1 if maximize else 0), _p(lb), _p(ub),
                                 C.byref(options) if options is not None else None, C.byref(status), C.byref(obj), _p(x),
                                 _p(of), _p(ot), _p(rf), _p(rt), _p(du)))
    return status.value, obj.value, x, of, ot, rf[:m], rt[:m], du[:m]


def solve_batch(A, b, c, lb=None, ub=None, sense=None, maximize=False, options: Options | None = None, out=None):
    """elp_solve_batch on host arrays.  `out` = (status int32[B], obj f64[B], x f64[B, n]) lets the caller supply the result
    buffers (e.g. page-locked ones, so the device->host copies of the streamed call stay asynchronous)."""
    A = _f64(A)
    B, m, n = A.shape
    b, c = _f64(b, (B, m)), _f64(c, (B, n))
    lb = _f64(lb, (B, n)) if lb is not None else None
    ub = _f64(ub, (B, n)) if ub is not None else None
    sense = _i8(np.broadcast_to(sense, (B, m))) if sense is not None else None
    if out is not None:
        status, obj, x = out
        assert status.dtype == np.int32 and status.shape == (B,) and status.flags.c_contiguous
        assert obj.dtype == np.float64 and obj.shape == (B,) and obj.flags.c_contiguous
        assert x.dtype == np.float64 and x.shape == (B, n) and x.flags.c_contiguous
    else:
        status = np.zeros(B, np.int32)
        obj = np.zeros(B)
        x = np.zeros((B, n))
    st = Stats()
    _check(lib().elp_solve_batch(C.c_int64(B), C.c_int32(m), C.c_int32(n), _p(A), _p(b), _p(c), _p(lb), _p(ub), _p(sense),
                                 C.c_int32(1 if maximize else 0), C.byref(options) if options is not None else None,
                                 _p(status), _p(obj), _p(x), C.byref(st)))
    return status, obj, x, st


class Batch:
    """Device-resident batch of dense LPs (inputs already in HBM; used by bench.py's `value` leg)."""

    def __init__(self, A, b, c, lb=None, ub=None, sense=None, maximize=False):
        A = _f64(A)
        self.B, self.m, self.n = A.shape
        B, m, n = A.shape
        b, c = _f64(b, (B, m)), _f64(c, (B, n))
        lb = _f64(lb, (B, n)) if lb is not None else None
        ub = _f64(ub, (B, n)) if ub is not None else None
        sense = _i8(np.broadcast_to(sense, (B, m))) if sense is not None else None
        self._h = C.c_void_p()
        _check(lib().elp_batch_create(C.c_int64(B), C.c_int32(m), C.c_int32(n), _p(A), _p(b), _p(c), _p(lb), _p(ub),
                                      _p(sense), C.c_int32(1 if maximize else 0), C.byref(self._h)))

    def run(self, options: Options | None = None) -> Stats:
        st = Stats()
        _check(lib().elp_batch_run(self._h, C.byref(options) if options is not None else None, C.byref(st)))
        return st

    def fetch(self):
        status = np.zeros(self.B, np.int32)
        obj = np.zeros(self.B)
        x = np.zeros((self.B, self.n))
        _check(lib().elp_batch_fetch(self._h, _p(status), _p(obj), _p(x)))
        return status, obj, x

    def close(self):
        if self._h:
            lib().elp_batch_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def spmv(m, n, row_ptr, col_idx, vals, x):
    out = np.zeros(m)
    _check(lib().elp_spmv(C.c_int32(m), C.c_int32(n), _p(_i32(row_ptr)), _p(_i32(col_idx)), _p(_f64(vals)), _p(_f64(x)),
                          _p(out)))
    return out


def check_feasible(m, n, row_ptr, col_idx, vals, x, sense, rhs, tol=2e-8):
    out = np.zeros(m, np.uint8)
    _check(lib().elp_check_feasible(C.c_int32(m), C.c_int32(n), _p(_i32(row_ptr)), _p(_i32(col_idx)), _p(_f64(vals)),
                                    _p(_f64(x)), _p(_i8(sense)), _p(_f64(rhs)), C.c_double(tol), _p(out)))
    return out.astype(bool)


class Pdlp:
    """Device-resident PDLP solver (optionally one row block of a distributed solve)."""

    def __init__(self, m, n, row_ptr, col_idx, vals, sense, rhs, c, lb, ub, maximize=False,
                 options: Options | None = None, dist=False):
        self.m, self.n = m, n
        row_ptr, col_idx = _i32(row_ptr), _i32(col_idx)
        self._h = C.c_void_p()
        self.setup_stats = Stats()
        _check(lib().elp_pdlp_create(C.c_int32(m), C.c_int32(n), _p(row_ptr), _p(col_idx), _p(_f64(vals)), _p(_i8(sense)),
                                     _p(_f64(rhs)), _p(_f64(c)), C.c_int32(1 if maximize else 0), _p(_f64(lb, (n,))),
                                     _p(_f64(ub, (n,))), C.byref(options) if options is not None else None,
                                     C.c_int32(1 if dist else 0), C.byref(self._h), C.byref(self.setup_stats)))

    def run(self, max_new_iters=0) -> Stats:
        st = Stats()
        _check(lib().elp_pdlp_run(self._h, C.c_int32(max_new_iters), C.byref(st)))
        return st

    def reset(self):
        _check(lib().elp_pdlp_reset(self._h))

    def solution(self):
        x = np.zeros(self.n)
        y = np.zeros(max(self.m, 1))
        obj = C.c_double()
        _check(lib().elp_pdlp_solution(self._h, _p(x), _p(y), C.byref(obj)))
        return x, y[:self.m], obj.value

    def probe_spmv(self, reps=20):
        a, b = C.c_double(), C.c_double()
        _check(lib().elp_pdlp_probe_spmv(self._h, C.c_int32(reps), C.byref(a), C.byref(b)))
        return a.value, b.value

    def probe_step(self, reps=20):
        a, b = C.c_double(), C.c_double()
        _check(lib().elp_pdlp_probe_step(self._h, C.c_int32(reps), C.byref(a), C.byref(b)))
        return a.value, b.value

    def transpose(self) -> int:
        """TRANSPOSE_GATHER or TRANSPOSE_SCATTER: how the plain iterations of this handle form A'y."""
        mode = C.c_int32(0)
        _check(lib().elp_pdlp_transpose(self._h, C.byref(mode)))
        return mode.value

    def close(self):
        if self._h:
            lib().elp_pdlp_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def comm_unique_id() -> bytes:
    buf = C.create_string_buffer(UNIQUE_ID_BYTES)
    _check(lib().elp_comm_unique_id(buf))
    return buf.raw


def comm_init(nranks: int, rank: int, uid: bytes):
    assert len(uid) == UNIQUE_ID_BYTES
    _check(lib().elp_comm_init(C.c_int32(nranks), C.c_int32(rank), C.create_string_buffer(uid, UNIQUE_ID_BYTES)))


def comm_destroy():
    _check(lib().elp_comm_destroy())
