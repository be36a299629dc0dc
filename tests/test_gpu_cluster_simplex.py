"""Simplex on a thread-block cluster (csrc/simplex.cu, simplex_kernel with C >= 2 CTAs): LPs, MILPs and sensitivity
ranging whose dense tableau [A | I] does not fit one SM's shared memory.  CPU: the C oracle agrees with HiGHS on every
family used below.  GPU: clusters forced onto shapes one CTA holds give the one-CTA instance's bytes (status, pivots,
basis-derived x and y, ranging); beyond one SM it agrees with the oracle and HiGHS; shapes beyond the largest cluster
are refused with an error naming the shape and the capacity; the AUTO size rule is unchanged."""
import numpy as np
import pytest

from easylp_b200 import _lib as L
from oracle import cbind, gen, ranging_ref

SMEM_MAX = 227 * 1024


def _up2(v):
    return (v + 1) & ~1


def auto_bytes(m, n):
    """ELP_METHOD_AUTO's footprint (simplex_auto_prefers: simplex when it is at most 200 KB)"""
    N = m + n
    d = _up2(m * n) + _up2(m * m) + _up2(m) + 4 * _up2(N) + _up2(m) + _up2(m) + _up2(N) + 8
    return d * 8 + 16 + ((m + 3) & ~3) * 4 + ((N + 3) & ~3) * 4 + 32


def cluster_bytes(m, n, C):
    """per-CTA shared memory of simplex_kernel with C CTAs per LP (SimplexLayout)"""
    w = (((m + n + C - 1) // C) + 1) & ~1
    d = m * w + 6 * _up2(m) + 5 * w + 8 + 16 + 16 + 4
    return d * 8 + 16 + ((m + 3) & ~3) * 4 + ((w + 3) & ~3) * 4 + 32 + 64 + 16


def expected_ctas(m, n, largest):
    if cluster_bytes(m, n, 1) <= SMEM_MAX:
        return 1
    for C in (2, 4, 8, 16):
        if C <= largest and cluster_bytes(m, n, C) <= SMEM_MAX:
            return C
    return None


def to_csr(A):
    m = A.shape[0]
    rp = np.zeros(m + 1, np.int32)
    ci, v = [], []
    for i in range(m):
        nz = np.nonzero(A[i])[0]
        ci += nz.tolist(); v += A[i, nz].tolist()
        rp[i + 1] = len(ci)
    return rp, np.array(ci, np.int32), np.array(v, float)


def planted(m, n, seed, kind="optimal"):
    """max c'x over A x <= b, x >= 0 with A >= 0 (every column has an entry), b = A x0 + slack: bounded and feasible.
    kind 'infeasible' adds a >= copy of row 0 beyond its <= right-hand side; 'unbounded' empties a column."""
    rng = np.random.default_rng(seed)
    A = rng.uniform(0.1, 1.0, size=(m, n)) * (rng.random((m, n)) < 0.4)
    A[rng.integers(0, m, n), np.arange(n)] = rng.uniform(0.2, 1.0, n)
    x0 = rng.uniform(0, 1, n) * (rng.random(n) < 0.5)
    rhs = A @ x0 + rng.uniform(0.1, 1.0, m)
    sense = np.zeros(m, np.int8)
    c = rng.uniform(0.1, 1.0, n)
    if kind == "infeasible":
        A[1] = A[0]
        rhs[1] = rhs[0] + 1.0
        sense[1] = L.GE
    if kind == "unbounded":
        A[:, n // 2] = 0.0
    rp, ci, v = to_csr(A)
    return dict(m=m, n=n, row_ptr=rp, col_idx=ci, vals=v, sense=sense, rhs=rhs, c=c, lb=np.zeros(n),
                ub=np.full(n, np.inf), maximize=True, A=A)


def mixed(m, n, seed):
    """mixed senses, equality rows, free and boxed variables.  seed % 4 picks the kind: 0 and 1 bounded (every variable
    boxed except the free ones, which carry no cost), 2 the same with two contradicting equality rows (infeasible),
    3 half the variables unbounded above with random costs (mostly unbounded)"""
    rng = np.random.default_rng(seed)
    kind = seed % 4
    A = np.round(rng.normal(size=(m, n)) * 2) / 2 * (rng.random((m, n)) < 0.3)
    x0 = np.round(rng.normal(size=n))
    sense = rng.choice([0, 0, 0, 1, 2], size=m).astype(np.int8)
    slack = np.round(rng.uniform(0, 3, size=m))
    rhs = A @ x0 + np.where(sense == 0, slack, np.where(sense == 1, -slack, 0.0))
    if kind == 2:                  # row 1 := row 0 as an equality one unit away from row 0's equality: infeasible
        A[1] = A[0]
        sense[0] = sense[1] = L.EQ
        rhs[1] = rhs[0] + 1.0
    c = np.round(rng.normal(size=n) * 2) / 2
    free = rng.random(n) < 0.2
    lb = np.where(free, -np.inf, np.minimum(x0, 0.0) - np.round(rng.random(n) * 2))
    ub = np.maximum(x0, 0.0) + np.round(rng.random(n) * 4)
    if kind == 3:
        ub = np.where(rng.random(n) < 0.5, np.inf, ub)
    else:
        c = np.where(free, 0.0, c)
    ub = np.where(free, np.inf, ub)
    rp, ci, v = to_csr(A)
    return dict(m=m, n=n, row_ptr=rp, col_idx=ci, vals=v, sense=sense, rhs=rhs, c=c, lb=lb, ub=ub,
                maximize=bool(rng.random() < 0.5), A=A)


def highs_lp(p):
    from scipy.optimize import linprog
    sign = -1.0 if p["maximize"] else 1.0
    A, s = p["A"], p["sense"]
    A_ub = np.vstack([A[s == 0], -A[s == 1]])
    b_ub = np.concatenate([p["rhs"][s == 0], -p["rhs"][s == 1]])
    r = linprog(sign * p["c"], A_ub=A_ub if A_ub.size else None, b_ub=b_ub if A_ub.size else None,
                A_eq=A[s == 2] if (s == 2).any() else None, b_eq=p["rhs"][s == 2] if (s == 2).any() else None,
                bounds=list(zip(p["lb"], p["ub"])), method="highs-ds")
    return {0: 0, 2: 2, 3: 3}.get(r.status, -1), (sign * r.fun if r.status == 0 else None)


def oracle_lp(p):
    return cbind.simplex_csr(p["m"], p["n"], p["row_ptr"], p["col_idx"], p["vals"], p["sense"], p["rhs"], p["c"], p["lb"],
                             p["ub"], maximize=p["maximize"])


def transport_20x40():
    p = gen.transport(20, 40, seed=3)
    A = np.zeros((p["m"], p["n"]))
    for i in range(p["m"]):
        A[i, p["col_idx"][p["row_ptr"][i]:p["row_ptr"][i + 1]]] = p["vals"][p["row_ptr"][i]:p["row_ptr"][i + 1]]
    p["A"] = A
    return p


def assignment(k, seed):
    rng = np.random.default_rng(seed)
    cost = rng.integers(1, 100, size=(k, k)).astype(float)
    n, m = k * k, 2 * k
    A = np.zeros((m, n))
    for i in range(k):
        A[i, i * k:(i + 1) * k] = 1.0            # worker i does one job
        A[k + i, i::k] = 1.0                     # job i gets one worker
    rp, ci, v = to_csr(A)
    return dict(m=m, n=n, row_ptr=rp, col_idx=ci, vals=v, sense=np.full(m, L.EQ, np.int8), rhs=np.ones(m), c=cost.ravel(),
                lb=np.zeros(n), ub=np.ones(n), is_integer=np.ones(n, np.uint8), maximize=False, A=A, cost=cost)


def random_milp(m, n, seed):
    rng = np.random.default_rng(seed)
    A = np.round(rng.uniform(0, 9, size=(m, n))) * (rng.random((m, n)) < 0.1)
    rhs = np.round(A.sum(axis=1) * rng.uniform(0.3, 0.6, size=m)) + 1.0
    c = np.round(rng.uniform(1, 20, size=n))
    is_int = (rng.random(n) < 0.05).astype(np.uint8)
    rp, ci, v = to_csr(A)
    return dict(m=m, n=n, row_ptr=rp, col_idx=ci, vals=v, sense=np.zeros(m, np.int8), rhs=rhs, c=c, lb=np.zeros(n),
                ub=np.full(n, 3.0), is_integer=is_int, maximize=True, A=A)


def random_ranging_lp(seed, m=120, n=300):
    """tests/test_sensitivity.py's random_lp, scaled up past one SM"""
    rng = np.random.default_rng(seed)
    A = rng.uniform(0.1, 3.0, size=(m, n)) * (rng.random((m, n)) < 0.8)
    A[:, 0] = rng.uniform(0.5, 2.0, size=m)
    x0 = rng.uniform(0.5, 3.0, size=n)
    rhs = A @ x0 + rng.uniform(0.1, 2.0, size=m)
    rp, ci, v = to_csr(A)
    return dict(m=m, n=n, row_ptr=rp, col_idx=ci, vals=v, sense=np.zeros(m, np.int8), rhs=rhs,
                c=rng.uniform(0.5, 4.0, size=n), lb=np.zeros(n), ub=np.full(n, 20.0), maximize=True, A=A)


BEYOND = [("transport", 60, 800), ("planted", 80, 300), ("planted", 200, 700), ("planted", 250, 700), ("planted", 100, 170)]


# ---- CPU: the oracle is sound at these sizes ---------------------------------------------------------------------------
@pytest.mark.parametrize("family", ["transport", "planted-80x300", "planted-200x700", "infeasible", "unbounded", "mixed"])
def test_oracle_agrees_with_highs_on_the_cluster_families(family):
    pytest.importorskip("scipy")
    if family == "transport":
        ps = [transport_20x40()]
    elif family == "planted-80x300":
        ps = [planted(80, 300, s) for s in range(2)]
    elif family == "planted-200x700":
        ps = [planted(200, 700, 7)]
    elif family == "infeasible":
        ps = [planted(80, 300, 11, "infeasible")]
    elif family == "unbounded":
        ps = [planted(80, 300, 12, "unbounded")]
    else:
        ps = [mixed(m, n, s) for (m, n) in [(40, 100), (60, 150), (90, 120)] for s in range(4)]
    for p in ps:
        st, obj, x, y, piv = oracle_lp(p)
        hs, hobj = highs_lp(p)
        assert st == hs, (p["m"], p["n"], st, hs)
        if st == 0:
            assert abs(obj - hobj) <= 1e-9 * max(1.0, abs(hobj))


def test_size_rule_places_the_issue_shapes():
    assert expected_ctas(40, 100, 16) == 1 and expected_ctas(90, 120, 16) == 1
    assert expected_ctas(60, 800, 16) == 2 and expected_ctas(80, 300, 16) == 2 and expected_ctas(50, 625, 16) == 2
    assert expected_ctas(200, 700, 16) == 8
    assert expected_ctas(250, 700, 16) == 16 and expected_ctas(250, 700, 8) is None
    assert expected_ctas(100, 150, 16) == 1 and expected_ctas(100, 170, 16) == 2


# ---- GPU ---------------------------------------------------------------------------------------------------------------
def _solve(p, monkeypatch, C=None, method=L.METHOD_SIMPLEX):
    if C is None:
        monkeypatch.delenv("ELP_SIMPLEX_CLUSTER", raising=False)
    else:
        monkeypatch.setenv("ELP_SIMPLEX_CLUSTER", str(C))
    return L.solve_lp(p["m"], p["n"], p["row_ptr"], p["col_idx"], p["vals"], p["sense"], p["rhs"], p["c"], p["lb"], p["ub"],
                      maximize=p["maximize"], options=L.default_options(method=method))


@pytest.fixture(scope="module")
def largest_cluster():
    """16 when the device schedules 16-CTA clusters of the largest footprint, else 8"""
    import os
    p = planted(40, 100, 0)
    old = os.environ.get("ELP_SIMPLEX_CLUSTER")
    os.environ["ELP_SIMPLEX_CLUSTER"] = "16"
    try:
        r = L.solve_lp(p["m"], p["n"], p["row_ptr"], p["col_idx"], p["vals"], p["sense"], p["rhs"], p["c"], p["lb"], p["ub"],
                       maximize=True, options=L.default_options(method=L.METHOD_SIMPLEX))
    finally:
        if old is None:
            del os.environ["ELP_SIMPLEX_CLUSTER"]
        else:
            os.environ["ELP_SIMPLEX_CLUSTER"] = old
    return 16 if r.stats.simplex_ctas == 16 else 8


def _cluster_sizes(largest):
    return [C for C in (2, 4, 8, 16) if C <= largest]


def _same_bits(a, b):
    return np.asarray(a).tobytes() == np.asarray(b).tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("m,n", [(40, 100), (60, 150), (90, 120)])
def test_forced_cluster_gives_the_one_cta_instances_bytes_through_solve_lp(m, n, monkeypatch, largest_cluster):
    statuses = set()
    for seed in range(12):
        p = mixed(m, n, 1000 * m + seed)
        ref = _solve(p, monkeypatch)
        assert ref.stats.simplex_ctas == 1
        statuses.add(ref.status)
        for C in _cluster_sizes(largest_cluster):
            r = _solve(p, monkeypatch, C)
            assert r.stats.simplex_ctas == C
            assert r.status == ref.status and r.stats.iterations == ref.stats.iterations, (seed, C)
            assert _same_bits(r.x, ref.x) and _same_bits(r.y, ref.y), (seed, C)
            if np.isfinite(ref.objval):
                assert abs(r.objval - ref.objval) <= 1e-12 * max(1.0, abs(ref.objval))
            else:
                assert r.objval == ref.objval
    assert 0 in statuses and len(statuses) >= 2


@pytest.mark.gpu
@pytest.mark.parametrize("m,n", [(40, 100), (90, 120)])
def test_forced_cluster_gives_the_one_cta_instances_bytes_through_solve_batch(m, n, monkeypatch, largest_cluster):
    ps = [mixed(m, n, 7 * m + s) for s in range(24)]
    A = np.stack([p["A"] for p in ps]); b = np.stack([p["rhs"] for p in ps]); c = np.stack([p["c"] for p in ps])
    lb = np.stack([p["lb"] for p in ps]); ub = np.stack([p["ub"] for p in ps]); sense = np.stack([p["sense"] for p in ps])
    c = np.where(np.array([p["maximize"] for p in ps])[:, None], -c, c)
    monkeypatch.delenv("ELP_SIMPLEX_CLUSTER", raising=False)
    s0, o0, x0, st0 = L.solve_batch(A, b, c, lb, ub, sense)
    assert st0.simplex_ctas == 1
    for C in _cluster_sizes(largest_cluster):
        monkeypatch.setenv("ELP_SIMPLEX_CLUSTER", str(C))
        s1, o1, x1, st1 = L.solve_batch(A, b, c, lb, ub, sense)
        assert st1.simplex_ctas == C and st1.iterations == st0.iterations
        assert _same_bits(s1, s0) and _same_bits(x1, x0)
        fin = np.isfinite(o0)
        assert np.array_equal(o1[~fin], o0[~fin])
        assert np.all(np.abs(o1[fin] - o0[fin]) <= 1e-12 * np.maximum(1.0, np.abs(o0[fin])))


@pytest.mark.gpu
def test_forced_cluster_gives_the_one_cta_instances_ranging(monkeypatch, largest_cluster):
    checked = 0
    for seed in range(6):
        p = random_ranging_lp(seed, m=40, n=100)
        monkeypatch.delenv("ELP_SIMPLEX_CLUSTER", raising=False)
        ref = L.sensitivity(p["m"], p["n"], p["row_ptr"], p["col_idx"], p["vals"], p["sense"], p["rhs"], p["c"], p["lb"],
                            p["ub"], maximize=True)
        for C in _cluster_sizes(largest_cluster):
            monkeypatch.setenv("ELP_SIMPLEX_CLUSTER", str(C))
            r = L.sensitivity(p["m"], p["n"], p["row_ptr"], p["col_idx"], p["vals"], p["sense"], p["rhs"], p["c"], p["lb"],
                              p["ub"], maximize=True)
            assert r[0] == ref[0]
            for a, b in zip(r[2:], ref[2:]):
                assert _same_bits(a, b)
        checked += ref[0] == 0
    assert checked >= 3


def _beyond_problem(kind, m, n, seed=7):
    return transport_20x40() if kind == "transport" else planted(m, n, seed)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,m,n", BEYOND)
def test_beyond_one_sm_against_the_oracle_and_highs(kind, m, n, monkeypatch, largest_cluster):
    p = _beyond_problem(kind, m, n)
    want = expected_ctas(m, n, largest_cluster)
    if want is None:
        with pytest.raises(L.ElpError, match=f"{m} x {n}"):
            _solve(p, monkeypatch)
        return
    r = _solve(p, monkeypatch)
    st, obj, x, y, piv = oracle_lp(p)
    hs, hobj = highs_lp(p)
    assert r.stats.simplex_ctas == want
    assert r.status == st == hs == 0
    assert abs(r.objval - obj) <= 1e-9 * max(1.0, abs(obj))
    assert abs(r.objval - hobj) <= 1e-9 * max(1.0, abs(hobj))
    ax = p["A"] @ r.x
    s = p["sense"]
    viol = np.where(s == L.LE, ax - p["rhs"], np.where(s == L.GE, p["rhs"] - ax, np.abs(ax - p["rhs"])))
    assert np.max(viol / np.maximum(1.0, np.abs(p["rhs"]))) <= 1e-7
    assert np.all(r.x >= -1e-9)
    # every bound is 0 / +inf: strong duality b'y = objective
    assert abs(float(p["rhs"] @ r.y) - r.objval) <= 1e-9 * max(1.0, abs(r.objval))


@pytest.mark.gpu
@pytest.mark.parametrize("kind,want_status", [("infeasible", L.STATUS_INFEASIBLE), ("unbounded", L.STATUS_UNBOUNDED)])
def test_beyond_one_sm_infeasible_and_unbounded(kind, want_status, monkeypatch):
    p = planted(80, 300, 11 if kind == "infeasible" else 12, kind)
    r = _solve(p, monkeypatch)
    st = oracle_lp(p)[0]
    hs, _ = highs_lp(p)
    assert r.stats.simplex_ctas == 2
    assert r.status == st == hs == want_status


@pytest.mark.gpu
def test_beyond_one_sm_through_the_device_resident_model(monkeypatch):
    from easylp_b200 import lower
    p = planted(80, 300, 5)
    rows = np.repeat(np.arange(p["m"]), np.diff(p["row_ptr"])).astype(np.int32)
    mdl = L.Model(rows, p["col_idx"], p["vals"], lower.pack([]), p["m"], p["n"])
    try:
        monkeypatch.delenv("ELP_SIMPLEX_CLUSTER", raising=False)
        r = mdl.solve(p["sense"], p["rhs"], p["c"], p["lb"], p["ub"], maximize=True,
                      options=L.default_options(method=L.METHOD_SIMPLEX))
    finally:
        mdl.close()
    ref = _solve(p, monkeypatch)
    assert r.stats.simplex_ctas == 2 and r.status == 0
    assert _same_bits(r.x, ref.x) and r.objval == ref.objval


@pytest.mark.gpu
def test_assignment_25x25_milp_beyond_one_sm(monkeypatch):
    from scipy.optimize import linear_sum_assignment
    monkeypatch.delenv("ELP_SIMPLEX_CLUSTER", raising=False)
    p = assignment(25, 4)
    r = L.solve_mip(p["m"], p["n"], p["row_ptr"], p["col_idx"], p["vals"], p["sense"], p["rhs"], p["c"], p["lb"], p["ub"],
                    p["is_integer"])
    ri, ci = linear_sum_assignment(p["cost"])
    assert r.status == 0 and r.stats.simplex_ctas == 2
    assert r.objval == p["cost"][ri, ci].sum()
    assert np.array_equal(r.x, np.round(r.x)) and np.array_equal(r.x.reshape(25, 25).sum(axis=1), np.ones(25))


# seeds whose trees stay small: the C oracle's branch and bound (oracle/mip_ref.py) solves them in 21, 7 and 11 nodes
MILP_SEEDS = [0, 1, 2]


@pytest.mark.gpu
@pytest.mark.parametrize("seed", MILP_SEEDS)
def test_random_milps_beyond_one_sm_against_highs(seed, monkeypatch):
    from scipy.optimize import Bounds, LinearConstraint, milp
    monkeypatch.delenv("ELP_SIMPLEX_CLUSTER", raising=False)
    p = random_milp(80, 300, seed)
    r = L.solve_mip(p["m"], p["n"], p["row_ptr"], p["col_idx"], p["vals"], p["sense"], p["rhs"], p["c"], p["lb"], p["ub"],
                    p["is_integer"], maximize=True, options=L.default_options(max_iter=20000))
    h = milp(-p["c"], constraints=LinearConstraint(p["A"], -np.inf, p["rhs"]), integrality=p["is_integer"].astype(int),
             bounds=Bounds(p["lb"], p["ub"]))
    assert r.stats.simplex_ctas == 2
    assert r.status == {0: 0, 2: 2, 3: 3}.get(h.status, -1), (r.status, h.status, r.stats.restarts)
    assert abs(r.objval - (-h.fun)) <= 1e-9 * max(1.0, abs(h.fun)), (r.objval, -h.fun, r.stats.restarts)
    print(f"seed {seed}: {r.stats.restarts} nodes, {r.stats.iterations} pivots")


def _nondegenerate(p, h):
    x = h["x"]
    slack = p["rhs"] - p["A"] @ x
    cb, rb = h["col_status"] == 0, h["row_status"] == 0
    ok = np.all((x[cb] > p["lb"][cb] + 1e-7) & (x[cb] < p["ub"][cb] - 1e-7)) and np.all(np.abs(slack[rb]) > 1e-7)
    return bool(ok) and int(cb.sum() + rb.sum()) == p["m"]


def _close(a, b, tol=1e-7):
    a, b = np.asarray(a, float), np.asarray(b, float)
    both_inf = np.isinf(a) & np.isinf(b) & (np.sign(a) == np.sign(b))
    return np.all(both_inf | (np.abs(a - b) <= tol * (1 + np.abs(b))))


@pytest.mark.gpu
def test_sensitivity_beyond_one_sm(monkeypatch):
    monkeypatch.delenv("ELP_SIMPLEX_CLUSTER", raising=False)
    checked = 0
    for seed in range(8):
        p = random_ranging_lp(seed)
        h = ranging_ref.highs(p)
        if h is None or not _nondegenerate(p, h):
            continue
        st, obj, x, of, ot, rf, rt, du = L.sensitivity(p["m"], p["n"], p["row_ptr"], p["col_idx"], p["vals"], p["sense"],
                                                       p["rhs"], p["c"], p["lb"], p["ub"], maximize=True)
        assert st == 0 and np.allclose(x, h["x"], atol=1e-8)
        # the restatement ranges HiGHS' basis at the simplex vertex: HiGHS' own x meets binding rows only to its
        # feasibility tolerance (5.7e-8 off at seed 6), which moves slacks out of the restatement's 1e-9 at-bound test
        rof, rot, rrf, rrt = ranging_ref.ranging(p, x, h["col_status"] == 0, h["row_status"] == 0)
        assert _close(of, rof) and _close(ot, rot) and _close(rf, rrf) and _close(rt, rrt)
        bc, br = h["col_status"] == 0, h["row_status"] != 0      # HiGHS' ranging: basic columns, binding rows
        assert _close(of[bc], h["cost_dn"][bc]) and _close(ot[bc], h["cost_up"][bc])
        assert _close(rf[br], h["row_dn"][br]) and _close(rt[br], h["row_up"][br])
        checked += 1
    assert checked >= 2


@pytest.mark.gpu
def test_beyond_the_largest_cluster_is_refused(monkeypatch):
    monkeypatch.delenv("ELP_SIMPLEX_CLUSTER", raising=False)
    p = planted(600, 2000, 1)
    args = (p["m"], p["n"], p["row_ptr"], p["col_idx"], p["vals"], p["sense"], p["rhs"], p["c"], p["lb"], p["ub"])
    msg = r"600 x 2000 model .* holds at most \d+ columns"
    with pytest.raises(L.ElpError, match=msg):
        L.solve_lp(*args, maximize=True, options=L.default_options(method=L.METHOD_SIMPLEX))
    with pytest.raises(L.ElpError, match=msg):
        L.solve_mip(*args, np.ones(p["n"], np.uint8), maximize=True)
    with pytest.raises(L.ElpError, match=msg):
        L.sensitivity(*args, maximize=True)


@pytest.mark.gpu
def test_auto_keeps_its_size_rule(monkeypatch):
    monkeypatch.delenv("ELP_SIMPLEX_CLUSTER", raising=False)
    p = transport_20x40()
    r = _solve(p, monkeypatch, method=L.METHOD_AUTO)
    assert r.stats.method_used == L.METHOD_PDLP and r.stats.simplex_ctas == 0
    small = planted(40, 100, 3)
    r = _solve(small, monkeypatch, method=L.METHOD_AUTO)
    assert r.stats.method_used == L.METHOD_SIMPLEX and r.stats.simplex_ctas == 1
    # the rule stays on its own footprint: 100 x 135 is below 200 KB there (not on the one-CTA footprint), 100 x 140 above
    assert auto_bytes(100, 135) <= 200 * 1024 < cluster_bytes(100, 135, 1) and auto_bytes(100, 140) > 200 * 1024
    r = _solve(planted(100, 135, 3), monkeypatch, method=L.METHOD_AUTO)
    assert r.stats.method_used == L.METHOD_SIMPLEX and r.stats.simplex_ctas == 1
    r = _solve(planted(100, 140, 3), monkeypatch, method=L.METHOD_AUTO)
    assert r.stats.method_used == L.METHOD_PDLP
