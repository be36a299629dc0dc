"""GPU parity tests for the three kernels, through the C ABI (ctypes).  Run on the B200 box."""
import numpy as np
import pytest

from easylp_b200 import _lib as L
from oracle import cbind, gen

pytestmark = pytest.mark.gpu


def _assemble_ref(row, col, val, m, n):
    """left-fold in emission order, drop zeros, row-major ascending col (what the dense reference yields)."""
    acc = {}
    for r, c, v in zip(row.tolist(), col.tolist(), val.tolist()):
        acc[(r, c)] = acc.get((r, c), 0.0) + v
    keys = sorted(k for k, v in acc.items() if v != 0.0)
    row_ptr = np.zeros(m + 1, np.int32)
    for r, _ in keys:
        row_ptr[r + 1] += 1
    row_ptr = np.cumsum(row_ptr).astype(np.int32)
    return row_ptr, np.array([c for _, c in keys], np.int32), np.array([acc[k] for k in keys])


@pytest.mark.parametrize("T,m,n,seed", [(0, 3, 4, 0), (1, 1, 1, 1), (50, 5, 7, 2), (5000, 40, 60, 3),
                                        (100_000, 300, 500, 4), (300_000, 2000, 100_000, 5)])
def test_assemble_bit_exact(T, m, n, seed):
    rng = np.random.default_rng(seed)
    row = rng.integers(0, m, size=T).astype(np.int32)
    col = rng.integers(0, max(n // 3, 1), size=T).astype(np.int32) * 3 % n
    val = rng.normal(size=T) * 10.0 ** rng.integers(-8, 8, size=T)
    if T > 10:
        # exact cancellations and duplicates
        row[1], col[1], val[1] = row[0], col[0], -val[0]
        row[5:9] = row[4]; col[5:9] = col[4]
    rp, ci, v, st = L.assemble_csr(row, col, val, m, n)
    rp0, ci0, v0 = _assemble_ref(row, col, val, m, n)
    assert np.array_equal(rp, rp0)
    assert np.array_equal(ci, ci0)
    assert v.tobytes() == v0.tobytes()          # bit-exact


def test_assemble_long_duplicate_run_order():
    # one key hit 10k times with values whose sum depends on the order
    rng = np.random.default_rng(7)
    T = 10_000
    val = rng.normal(size=T) * 10.0 ** rng.integers(-10, 10, size=T)
    row = np.zeros(T, np.int32); col = np.full(T, 2, np.int32)
    rp, ci, v, _ = L.assemble_csr(row, col, val, 1, 5)
    s = 0.0
    for t in val.tolist():
        s += t
    assert ci.tolist() == [2] and v[0] == s


@pytest.mark.parametrize("T,m,n,seed", [(5000, 40, 60, 3), (200_000, 3000, 5000, 8)])
def test_assemble_already_ordered_stream_skips_the_sort(T, m, n, seed, monkeypatch):
    """`$con()` emits row after row and most bodies walk their columns upwards: the stream arrives in (row, col) order, with
    duplicates adjacent in emission order.  The device detects that and skips the radix sort; same bits either way."""
    rng = np.random.default_rng(seed)
    row = rng.integers(0, m, size=T).astype(np.int32)
    col = rng.integers(0, n, size=T).astype(np.int32)
    val = rng.normal(size=T) * 10.0 ** rng.integers(-8, 8, size=T)
    order = np.lexsort((col, row))                       # stable: equal (row, col) keep their emission order
    row, col, val = row[order], col[order], val[order]
    rp0, ci0, v0 = _assemble_ref(row, col, val, m, n)
    rp, ci, v, st_fast = L.assemble_csr(row, col, val, m, n)
    assert np.array_equal(rp, rp0) and np.array_equal(ci, ci0) and v.tobytes() == v0.tobytes()
    monkeypatch.setenv("ELP_ASM_ALWAYS_SORT", "1")
    rp2, ci2, v2, st_sort = L.assemble_csr(row, col, val, m, n)
    assert np.array_equal(rp2, rp0) and np.array_equal(ci2, ci0) and v2.tobytes() == v0.tobytes()
    assert st_fast.kernel_launches < st_sort.kernel_launches


def _stream(kind, rng):
    if kind == "random":            # ~150 terms per row, columns spread, duplicates and cancellations
        T, m, n = 300_000, 2000, 100_000
        row = rng.integers(0, m, T); col = rng.integers(0, n, T)
    elif kind == "duplicates":      # few distinct columns: long equal-key runs whose sums depend on the order
        T, m, n = 120_000, 700, 40
        row = rng.integers(0, m, T); col = rng.integers(0, n, T)
    elif kind == "empty_rows":      # most rows have no term at all
        T, m, n = 50_000, 100_000, 3000
        row = rng.integers(0, m, T) // 7 * 7; col = rng.integers(0, n, T)
    elif kind == "one_column":
        T, m, n = 30_000, 5000, 1
        row = rng.integers(0, m, T); col = np.zeros(T, np.int64)
    elif kind == "long_rows_fit":   # one row per bucket, ~1300 terms each, ranked quadratically
        T, m, n = 2600, 2, 900
        row = np.arange(T) % 2; col = rng.integers(0, n, T)
    elif kind == "wide":            # 31 column bits leave one bit for the row inside a bucket
        T, m, n = 50_000, 1000, 2_000_000_000
        row = rng.integers(0, m, T); col = rng.integers(0, n, T)
    elif kind == "skewed":          # one row holds more terms than a bucket: the call falls back to the radix sort
        T, m, n = 60_000, 3000, 5000
        row = rng.integers(0, m, T); row[: T // 3] = 17; col = rng.integers(0, n, T)
    val = rng.normal(size=T) * 10.0 ** rng.integers(-8, 8, size=T)
    row = row.astype(np.int32); col = col.astype(np.int32)
    row[1], col[1], val[1] = row[0], col[0], -val[0]          # an exact cancellation
    return row, col, val, m, n


@pytest.mark.parametrize("kind", ["random", "duplicates", "empty_rows", "one_column", "long_rows_fit", "wide", "skewed"])
def test_assemble_bucketed_equals_sorted(kind, monkeypatch):
    """Unordered streams are split into row buckets that one CTA sorts and folds in shared memory (bucket_sort.cuh); the
    stable radix sort stays for streams with a bucket that does not fit.  Same bits as the sort and as the left fold of
    /root/reference/R/methods.R:248-250 restated on the host."""
    row, col, val, m, n = _stream(kind, np.random.default_rng(11))
    rp, ci, v, st_b = L.assemble_csr(row, col, val, m, n)
    monkeypatch.setenv("ELP_ASM_BUCKETED", "0")
    rp2, ci2, v2, st_s = L.assemble_csr(row, col, val, m, n)
    assert np.array_equal(rp, rp2) and np.array_equal(ci, ci2) and v.tobytes() == v2.tobytes()
    rp0, ci0, v0 = _assemble_ref(row, col, val, m, n)
    assert np.array_equal(rp, rp0) and np.array_equal(ci, ci0) and v.tobytes() == v0.tobytes()
    if kind == "skewed":
        assert st_b.kernel_launches > st_s.kernel_launches          # tried the buckets, then sorted
    else:
        assert st_b.kernel_launches < st_s.kernel_launches


def test_assemble_bucketed_is_deterministic():
    # the order inside a bucket depends on the atomics of the split; the ranking by (col, stream index) removes it
    row, col, val, m, n = _stream("duplicates", np.random.default_rng(5))
    a = L.assemble_csr(row, col, val, m, n)
    for _ in range(3):
        b = L.assemble_csr(row, col, val, m, n)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and a[2].tobytes() == b[2].tobytes()


def test_assemble_ordered_stream_row_pointers_across_empty_tiles():
    """Ordered path (assemble.cu: asm_ordered_count / _emit): row pointers are written by the surviving entries themselves,
    each starting the rows since its predecessor.  Stretches of the stream in which nothing survives (cancelling pairs over
    many tiles of 256 terms), empty rows in front, between and behind, and a stream in which nothing survives at all."""
    rng = np.random.default_rng(3)
    m, n = 5000, 700
    # rows 10..19 carry entries, 20..2999 nothing, 3000 carries 40 000 terms that cancel pairwise, 3001..4000 entries again
    row = np.concatenate([np.repeat(np.arange(10, 20), 30), np.full(40_000, 3000), np.repeat(np.arange(3001, 4001), 5)])
    col = np.concatenate([np.tile(np.arange(30) * 3, 10), np.repeat(np.arange(100), 400), np.tile(np.arange(5) * 7, 1000)])
    val = rng.normal(size=row.size)
    blk = slice(300, 40_300)
    v = val[blk].reshape(100, 400)
    v[:, 1::2] = -v[:, 0::2]                        # every (row 3000, col) run: x, -x, y, -y, ... folds to exactly 0
    val[blk] = v.ravel()
    row = row.astype(np.int32); col = col.astype(np.int32)
    assert np.all(np.diff(row.astype(np.int64) * n + col) >= 0)
    rp, ci, vv, st = L.assemble_csr(row, col, val, m, n)
    rp0, ci0, v0 = _assemble_ref(row, col, val, m, n)
    assert np.array_equal(rp, rp0) and np.array_equal(ci, ci0) and vv.tobytes() == v0.tobytes()
    assert rp[3000] == rp[3001] == 300                  # the cancelled row is empty
    # nothing survives at all
    rp, ci, vv, _ = L.assemble_csr(row[blk], col[blk], val[blk], m, n)
    assert ci.size == 0 and not rp.any()


def test_assemble_rejects_out_of_range():
    with pytest.raises(L.ElpError):
        L.assemble_csr([0, 5], [0, 0], [1.0, 1.0], 2, 2)


@pytest.mark.parametrize("order", ["ordered", "unordered"])
@pytest.mark.parametrize("what", ["row_high", "row_negative", "col_high"])
def test_assemble_rejects_out_of_range_in_long_streams(order, what):
    # every path (two-pass ordered, buckets, radix sort) reports the term and never uses it as an index; the library
    # stays usable afterwards
    rng = np.random.default_rng(2)
    T, m, n = 6000, 50, 40
    row = np.sort(rng.integers(0, m, T)).astype(np.int32)
    col = rng.integers(0, n, T).astype(np.int32)
    o = np.lexsort((col, row))
    row, col = row[o], col[o]
    val = rng.normal(size=T)
    if what == "row_high":
        row[-1] = 2_000_000_000
    elif what == "row_negative":
        row[0] = -7
    else:
        col[T // 2] = n
    if order == "unordered":
        p = rng.permutation(T)
        row, col, val = row[p], col[p], val[p]
    with pytest.raises(L.ElpError):
        L.assemble_csr(row, col, val, m, n)
    rp, ci, v, _ = L.assemble_csr([0, 1], [1, 0], [1.0, 2.0], 2, 2)
    assert rp.tolist() == [0, 1, 2] and ci.tolist() == [1, 0] and v.tolist() == [1.0, 2.0]


def test_spmv_and_feasible():
    p = gen.sparse_planted(3000, seed=1)
    x = np.random.default_rng(0).normal(size=p["n"])
    out = L.spmv(p["m"], p["n"], p["row_ptr"], p["col_idx"], p["vals"], x)
    # S4 is BIT-identical to a scalar loop (DESIGN 2): one lane per row, products and sums in index order, no FMA.
    # numpy float64 scalars do the same IEEE multiply / add one at a time (reduceat would sum pairwise).
    rp, ci, v = p["row_ptr"], p["col_idx"], p["vals"]
    ref = np.zeros(p["m"])
    for i in range(p["m"]):
        s = np.float64(0.0)
        for k in range(rp[i], rp[i + 1]):
            s = s + v[k] * x[ci[k]]
        ref[i] = s
    assert out.tobytes() == ref.tobytes()
    feas = L.check_feasible(p["m"], p["n"], p["row_ptr"], p["col_idx"], p["vals"], p["x_opt"], p["sense"], p["rhs"])
    assert feas.all()


def test_readme_lp_simplex():
    p = gen.readme_lp()
    r = L.solve_lp(p["m"], p["n"], p["row_ptr"], p["col_idx"], p["vals"], p["sense"], p["rhs"], p["c"], p["lb"], p["ub"],
                   maximize=True)
    assert r.status == 0 and r.status_string == "optimal"
    assert abs(r.objval - 2.0) < 1e-9 and np.allclose(r.x, [1.0, 1.0], atol=1e-9)
    assert r.stats.method_used == L.METHOD_SIMPLEX


def test_unbounded_no_rows():
    # /root/reference/tests/testthat/test-unbounded.R: max x, x free, no rows
    r = L.solve_lp(0, 1, [0], [], [], [], [], [1.0], [-np.inf], [np.inf], maximize=True)
    assert r.status == 3 and r.objval == np.inf and r.x[0] == np.inf


def test_batch_simplex_vs_oracle():
    d = gen.dense_batch(B=4000, seed=11)
    status, obj, x, st = L.solve_batch(d["A"], d["b"], d["c"], d["lb"], d["ub"], d["sense"])
    s0, o0, x0, piv = cbind.simplex_batch(d["A"], d["b"], d["c"], d["lb"], d["ub"], d["sense"], nthreads=8)
    assert np.array_equal(status, s0)
    assert np.all(np.abs(obj - o0) <= 1e-6 * np.maximum(1.0, np.abs(o0)))
    # primal feasibility of the returned points
    ax = np.einsum("bij,bj->bi", d["A"], x)
    assert np.all(ax <= d["b"] + 1e-7) and np.all(x >= -1e-9) and np.all(x <= 10 + 1e-9)


def test_batch_mixed_senses_free_vars():
    rng = np.random.default_rng(5)
    B, m, n = 3000, 6, 7
    A = np.round(rng.normal(size=(B, m, n)) * 2) / 2 * (rng.random((B, m, n)) < 0.7)
    b = np.round(rng.normal(size=(B, m)) * 4) / 2
    sense = rng.integers(0, 3, size=(B, m)).astype(np.int8)
    c = np.round(rng.normal(size=(B, n)) * 2) / 2
    lb = np.where(rng.random((B, n)) < 0.5, -np.inf, np.round(rng.normal(size=(B, n))))
    ub = np.where(rng.random((B, n)) < 0.5, np.inf, np.where(np.isfinite(lb), lb, 0.0) + np.round(rng.random((B, n)) * 4))
    status, obj, x, _ = L.solve_batch(A, b, c, lb, ub, sense)
    s0, o0, x0, _ = cbind.simplex_batch(A, b, c, lb, ub, sense, nthreads=8)
    assert np.array_equal(status, s0)
    ok = status == 0
    assert ok.sum() > 100 and (status == 2).sum() > 100 and (status == 3).sum() > 100
    assert np.all(np.abs(obj[ok] - o0[ok]) <= 1e-6 * np.maximum(1.0, np.abs(o0[ok])))


def _pdlp_check(p, eps=1e-6, **kw):
    r = L.solve_lp(p["m"], p["n"], p["row_ptr"], p["col_idx"], p["vals"], p["sense"], p["rhs"], p["c"], p["lb"], p["ub"],
                   maximize=p["maximize"], options=L.default_options(method=L.METHOD_PDLP, **kw))
    return r


def test_pdlp_readme():
    p = gen.readme_lp()
    r = _pdlp_check(p)
    assert r.status == 0 and abs(r.objval - 2.0) <= 1e-5
    assert r.stats.rel_primal_res <= 1e-6 and r.stats.rel_dual_res <= 1e-6 and r.stats.rel_gap <= 1e-6


@pytest.mark.parametrize("graph", [0, 1])
def test_pdlp_planted(graph):
    p = gen.sparse_planted(2000, seed=0)
    r = _pdlp_check(p, use_graph=graph)
    assert r.status == 0
    assert abs(r.objval - p["obj_opt"]) <= 1e-5 * max(1.0, abs(p["obj_opt"]))
    assert r.stats.rel_primal_res <= 1e-6 and r.stats.rel_dual_res <= 1e-6 and r.stats.rel_gap <= 1e-6


def _pdlp_handle(p, **kw):
    return L.Pdlp(p["m"], p["n"], p["row_ptr"], p["col_idx"], p["vals"], p["sense"], p["rhs"], p["c"], p["lb"], p["ub"],
                  maximize=p["maximize"], options=L.default_options(method=L.METHOD_PDLP, **kw))


@pytest.mark.parametrize("size,seed", [(300, 1), (5000, 2), (40000, 3)])
def test_pdlp_scatter_iterate_matches_gather(size, seed):
    """The scatter formulation (dual kernel leaves g = A'y behind by fp64 reductions, gather-free primal update) and
    the CSC-gather formulation are the same iteration: after a fixed number of PDHG iterations (two graph-replayed
    chunks + three checks) the candidates T(z) agree to rounding — only the summation order inside g differs."""
    p = gen.sparse_planted(size, seed=seed)
    out = {}
    for mode in (L.TRANSPOSE_GATHER, L.TRANSPOSE_SCATTER):
        h = _pdlp_handle(p, transpose=mode)
        assert h.transpose() == mode
        st = h.run(129)
        assert st.iterations == 129
        out[mode] = h.solution() + (st,)
        h.close()
    xg, yg, og, sg = out[L.TRANSPOSE_GATHER]
    xs, ys, os_, ss = out[L.TRANSPOSE_SCATTER]
    assert sg.restarts == ss.restarts
    assert np.max(np.abs(xg - xs)) <= 1e-9 * max(1.0, np.max(np.abs(xg)))
    assert np.max(np.abs(yg - ys)) <= 1e-9 * max(1.0, np.max(np.abs(yg)))
    assert abs(og - os_) <= 1e-9 * max(1.0, abs(og))


@pytest.mark.parametrize("mode", [1, 2])
@pytest.mark.parametrize("make", ["planted", "transport", "long_rows"])
def test_pdlp_transpose_modes_solve(mode, make):
    """both formulations reach the same optimum (status exact, objective 1e-6 relative, residuals <= 1e-6);
    'long_rows' has rows longer than a stage, which the scatter epilogue walks from global memory"""
    if make == "planted":
        p = gen.sparse_planted(3000, seed=7)
        ref = p["obj_opt"]
    elif make == "transport":
        p = gen.transport(12, 15, seed=3)
        st, ref, *_ = cbind.simplex_csr(p["m"], p["n"], p["row_ptr"], p["col_idx"], p["vals"], p["sense"], p["rhs"],
                                        p["c"], p["lb"], p["ub"])
        assert st == 0
    else:
        p = gen.transport(3, 700, seed=5)          # supply rows with 700 entries each
        st, ref, *_ = cbind.simplex_csr(p["m"], p["n"], p["row_ptr"], p["col_idx"], p["vals"], p["sense"], p["rhs"],
                                        p["c"], p["lb"], p["ub"])
        assert st == 0
    r = _pdlp_check(p, transpose=mode)
    assert r.status == 0
    assert abs(r.objval - ref) <= 2e-6 * max(1.0, abs(ref))
    assert r.stats.rel_primal_res <= 1e-6 and r.stats.rel_dual_res <= 1e-6 and r.stats.rel_gap <= 1e-6


def test_pdlp_transport_vs_simplex_oracle():
    p = gen.transport(12, 15, seed=3)
    r = _pdlp_check(p)
    st, obj, x, y, piv = cbind.simplex_csr(p["m"], p["n"], p["row_ptr"], p["col_idx"], p["vals"], p["sense"], p["rhs"],
                                           p["c"], p["lb"], p["ub"])
    assert st == 0 and r.status == 0
    assert abs(r.objval - obj) <= 2e-6 * max(1.0, abs(obj))


@pytest.mark.parametrize("m,n", [(1, 1), (2, 2), (3, 5), (4, 4), (7, 9), (8, 20), (12, 50), (16, 16), (20, 30), (24, 40),
                                 (28, 30), (32, 60), (5, 70), (10, 86), (33, 10), (20, 80), (40, 100)])
def test_batch_shapes_vs_oracle(m, n):
    """every register-tableau instantiation (rows padded to 4, 1-3 columns per lane), odd sizes (no TMA path) and
    the shapes that run one LP per CTA"""
    rng = np.random.default_rng(100 * m + n)
    B = 300
    A = rng.uniform(-0.3, 1.0, size=(B, m, n)) * (rng.random((B, m, n)) < 0.8)
    x0 = rng.uniform(0, 1, size=(B, n))
    b = np.einsum("bij,bj->bi", A, x0) + rng.uniform(0.1, 1.0, size=(B, m))
    sense = (rng.random((B, m)) < 0.15).astype(np.int8)            # mostly <=, some >=
    b = np.where(sense == 1, b - 2.0, b)
    c = rng.normal(size=(B, n))
    lb = np.zeros((B, n)); ub = np.full((B, n), 5.0)
    ub[:, ::3] = np.inf
    status, obj, x, _ = L.solve_batch(A, b, c, lb, ub, sense)
    s0, o0, x0_, _ = cbind.simplex_batch(A, b, c, lb, ub, sense, nthreads=8)
    assert np.array_equal(status, s0)
    ok = status == 0
    assert ok.sum() > 0
    assert np.all(np.abs(obj[ok] - o0[ok]) <= 1e-6 * np.maximum(1.0, np.abs(o0[ok])))
    ax = np.einsum("bij,bj->bi", A[ok], x[ok])
    viol = np.where(sense[ok] == 0, ax - b[ok], b[ok] - ax)
    assert viol.max() <= 1e-6


def test_batch_duals_small():
    """duals of the batched path on the README LP (y from the slack block of the final tableau)"""
    p = gen.readme_lp()
    r = L.solve_lp(p["m"], p["n"], p["row_ptr"], p["col_idx"], p["vals"], p["sense"], p["rhs"], p["c"], p["lb"], p["ub"],
                   maximize=True)
    # strong duality: b'y == objective
    assert abs(float(np.dot(p["rhs"], r.y)) - 2.0) <= 1e-9
