"""The plain single-GPU PDLP iterations stream only what the problem needs: x-bar is carried in place of x, bounds that
are the same constant in every column (l = +0.0, u = +inf) are not streamed, and the row bounds are rebuilt from the
scaled right-hand side and a sense byte.  Every specialisation must reach the oracle's optimum, and stopping and
resuming a solve anywhere must not change a bit of it."""
import numpy as np
import pytest

from easylp_b200 import _lib as L
from oracle import cbind, gen

pytestmark = pytest.mark.gpu


def _handle(p, **kw):
    return L.Pdlp(p["m"], p["n"], p["row_ptr"], p["col_idx"], p["vals"], p["sense"], p["rhs"], p["c"], p["lb"], p["ub"],
                  maximize=p["maximize"], options=L.default_options(method=L.METHOD_PDLP, **kw))


def _solve(p, **kw):
    h = _handle(p, **kw)
    st = h.run()
    x, y, obj = h.solution()
    h.close()
    return st, x, y, obj


def _general_bounds(m, seed):
    """planted LP with mixed bounds: -0.0, finite and infinite lower bounds, finite and infinite upper bounds.  Columns
    with a positive reduced cost stay at their bound 0 (+0.0 or -0.0), so the planted pair stays optimal."""
    p = gen.sparse_planted(m, seed=seed)
    rng = np.random.default_rng(seed + 100)
    n = p["n"]
    basic = p["x_opt"] > 0
    lb = np.zeros(n)
    lb[~basic & (rng.random(n) < 0.5)] = -0.0
    pick = rng.integers(0, 3, size=n)
    lb[basic & (pick == 0)] = -np.inf
    lb[basic & (pick == 1)] = -1.0
    lb[basic & (pick == 2)] = -0.0
    ub = np.where(rng.random(n) < 0.5, np.inf, 1e3)
    p["lb"], p["ub"] = lb, ub
    return p


def _planted(kind):
    if kind == "l0_ufinite":                      # the C4 generator: 0 <= x <= 1e3
        return gen.sparse_planted(3000, seed=11)
    if kind == "l0_uinf":
        return gen.sparse_planted(3000, seed=12, ub_val=np.inf)
    return _general_bounds(3000, seed=13)


@pytest.mark.parametrize("kind", ["l0_ufinite", "l0_uinf", "general"])
def test_bound_specialisations_solve(kind):
    p = _planted(kind)
    assert set(np.unique(p["sense"]).tolist()) == {L.LE, L.GE, L.EQ}
    if kind == "general":
        assert np.any(np.signbit(p["lb"]) & (p["lb"] == 0)) and np.isinf(p["lb"]).any() and np.isinf(p["ub"]).any()
    st, x, y, obj = _solve(p)
    assert st.status == 0
    assert abs(obj - p["obj_opt"]) <= 1e-5 * max(1.0, abs(p["obj_opt"]))
    assert st.rel_primal_res <= 1e-6 and st.rel_dual_res <= 1e-6 and st.rel_gap <= 1e-6
    assert np.all(x >= p["lb"] - 1e-9) and np.all(x <= p["ub"] + 1e-9)


def test_transport_l0_uinf_vs_simplex_oracle():
    p = gen.transport(12, 15, seed=3)
    assert np.all(p["lb"] == 0) and np.all(np.isinf(p["ub"]))
    st, x, y, obj = _solve(p)
    s0, o0, *_ = cbind.simplex_csr(p["m"], p["n"], p["row_ptr"], p["col_idx"], p["vals"], p["sense"], p["rhs"], p["c"],
                                   p["lb"], p["ub"])
    assert s0 == 0 and st.status == 0
    assert abs(obj - o0) <= 2e-6 * max(1.0, abs(o0))


def test_wide_lane_plan_keeps_row_bounds(monkeypatch):
    """eight lanes per row: tiles of four rows cannot carry a sense byte per row in 16-byte copies, so the dual
    epilogue keeps the lc / uc streams — and gives the same optimum"""
    monkeypatch.setenv("ELP_SPMV_L", "8")
    p = _general_bounds(2000, seed=21)
    st, x, y, obj = _solve(p)
    assert st.status == 0
    assert abs(obj - p["obj_opt"]) <= 1e-5 * max(1.0, abs(p["obj_opt"]))
    assert st.rel_primal_res <= 1e-6 and st.rel_dual_res <= 1e-6 and st.rel_gap <= 1e-6


def _first_restart(p):
    """iteration count right after the first restart (one iteration per run() call)"""
    h = _handle(p)
    try:
        for _ in range(20000):
            st = h.run(1)
            if st.restarts > 0:
                return st.iterations
            assert st.status == L.STATUS_TIMEOUT, "solved before the first restart"
    finally:
        h.close()
    raise AssertionError("no restart within 20000 iterations")


@pytest.mark.parametrize("kind", ["l0_ufinite", "general"])
def test_chunked_run_is_bit_identical(kind):
    """A solve stopped after 1, 63, 64, 65 iterations and right after the first restart, then resumed, takes the path of
    one uninterrupted solve bit for bit: x-bar carried through a stop, x stored by the last iteration of every chunk,
    graph and stream launches of the plain iterations, and the restart all agree."""
    p = _planted(kind)
    st_ref, x_ref, y_ref, obj_ref = _solve(p)
    assert st_ref.status == 0
    r = _first_restart(p)
    stops = sorted({1, 63, 64, 65, r, r + 1})
    h = _handle(p)
    done = 0
    for s in stops:
        st = h.run(s - done)
        assert st.iterations == s
        done = s
    st = h.run()
    x, y, obj = h.solution()
    h.close()
    assert st.status == st_ref.status and st.iterations == st_ref.iterations and st.restarts == st_ref.restarts
    assert x.tobytes() == x_ref.tobytes()
    assert y.tobytes() == y_ref.tobytes()
    assert np.float64(obj).tobytes() == np.float64(obj_ref).tobytes()


def test_probe_step_leaves_the_solve_unchanged():
    """probe_step times plain iterations from a mid-solve iterate and resets the handle; a solve after it is the same"""
    p = _planted("l0_ufinite")
    st_ref, x_ref, y_ref, _ = _solve(p)
    h = _handle(p)
    h.probe_step(5)
    st = h.run()
    x, y, _ = h.solution()
    h.close()
    assert st.iterations == st_ref.iterations
    assert x.tobytes() == x_ref.tobytes() and y.tobytes() == y_ref.tobytes()
