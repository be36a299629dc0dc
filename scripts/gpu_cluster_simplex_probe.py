"""Simplex on a thread-block cluster: per-pivot cost of the cluster kernel on medium LPs, against PDLP to 1e-6 on the same
LP, HiGHS' dual simplex on one CPU core (a stand-in for lp_solve, which is not available here) and branch and bound on
MILPs beyond one SM; forced clusters against the one-CTA instance on a shape one SM holds.

    python scripts/gpu_cluster_simplex_probe.py [out.json]

Device times are CUDA events around densify + simplex kernel (stats.solve_ms), the median of 3 solves after a warm-up.
Only one barrier style is built (cooperative_groups cluster.sync: barrier.cluster.arrive.release / wait.acquire)."""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import numpy as np

from easylp_b200 import _lib as L
import test_gpu_cluster_simplex as T


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:      # noqa: BLE001
        return f"nvidia-smi unavailable: {e}"


def set_cluster(C):
    if C is None:
        os.environ.pop("ELP_SIMPLEX_CLUSTER", None)
    else:
        os.environ["ELP_SIMPLEX_CLUSTER"] = str(C)


def solve(p, method=L.METHOD_SIMPLEX, C=None, reps=3):
    set_cluster(C)
    try:
        runs = []
        for _ in range(reps + 1):
            r = L.solve_lp(p["m"], p["n"], p["row_ptr"], p["col_idx"], p["vals"], p["sense"], p["rhs"], p["c"], p["lb"],
                           p["ub"], maximize=p["maximize"], options=L.default_options(method=method, eps_rel=1e-6))
            runs.append(r)
        runs = runs[1:]
        ms = sorted(r.stats.solve_ms for r in runs)[len(runs) // 2]
        wall = sorted(r.stats.total_ms for r in runs)[len(runs) // 2]
        return runs[0], ms, wall
    finally:
        set_cluster(None)


def highs_ms(p):
    from scipy.optimize import linprog
    sign = -1.0 if p["maximize"] else 1.0
    A, s = p["A"], p["sense"]
    t = time.perf_counter()
    r = linprog(sign * p["c"], A_ub=np.vstack([A[s == 0], -A[s == 1]]),
                b_ub=np.concatenate([p["rhs"][s == 0], -p["rhs"][s == 1]]), bounds=list(zip(p["lb"], p["ub"])),
                method="highs-ds")
    return (time.perf_counter() - t) * 1e3, (sign * r.fun if r.status == 0 else None)


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    res = {"gpu": gpu_info(), "lps": [], "mip": [], "cluster_vs_cta": []}
    p16 = T.planted(40, 100, 0)
    largest = 16 if solve(p16, C=16, reps=1)[0].stats.simplex_ctas == 16 else 8
    res["largest_cluster"] = largest
    shapes = [("transport 20x40", T.transport_20x40()), ("planted 150x400", T.planted(150, 400, 1)),
              ("planted 250x700", T.planted(250, 700, 2))]
    shapes.append(("largest: planted 300x1100", T.planted(300, 1100, 3)) if largest == 16
                  else ("largest: planted 200x850", T.planted(200, 850, 3)))
    for name, p in shapes:
        row = {"shape": name, "m": p["m"], "n": p["n"]}
        try:
            r, ms, wall = solve(p)
            row.update(C=r.stats.simplex_ctas, status=r.status, pivots=r.stats.iterations, device_ms=ms, wall_ms=wall,
                       us_per_pivot=ms * 1e3 / max(r.stats.iterations, 1), obj=r.objval)
        except L.ElpError as e:
            row.update(error=str(e))
        rp, pms, pwall = solve(p, method=L.METHOD_PDLP)
        row.update(pdlp_status=rp.status, pdlp_iters=rp.stats.iterations, pdlp_device_ms=pms, pdlp_wall_ms=pwall,
                   pdlp_obj=rp.objval)
        hm, hobj = highs_ms(p)
        row.update(highs_ds_one_core_ms=hm, highs_obj=hobj)
        res["lps"].append(row)
        print(json.dumps(row), flush=True)
    # branch and bound beyond one SM
    for name, p in [("assignment 25x25", T.assignment(25, 4))] + [(f"random milp 80x300 seed {s}", T.random_milp(80, 300, s))
                                                                  for s in T.MILP_SEEDS]:
        t = time.perf_counter()
        r = L.solve_mip(p["m"], p["n"], p["row_ptr"], p["col_idx"], p["vals"], p["sense"], p["rhs"], p["c"], p["lb"], p["ub"],
                        p["is_integer"], maximize=p["maximize"], options=L.default_options(max_iter=20000))
        wall = (time.perf_counter() - t) * 1e3
        row = dict(model=name, C=r.stats.simplex_ctas, status=r.status, obj=r.objval, nodes=r.stats.restarts,
                   pivots=r.stats.iterations, device_ms=r.stats.solve_ms, wall_ms=wall,
                   nodes_per_s=r.stats.restarts / (wall / 1e3))
        res["mip"].append(row)
        print(json.dumps(row), flush=True)
    # forced clusters against the one-CTA instance on shapes one SM holds
    for (m, n) in [(90, 120), (60, 150)]:
        p = T.mixed(m, n, 5)
        p["maximize"] = False
        base = None
        for C in [None] + [c for c in (2, 4, 8, 16) if c <= largest]:
            r, ms, _ = solve(p, C=C)
            if base is None:
                base = r
            row = dict(m=m, n=n, forced=C, C=r.stats.simplex_ctas, status=r.status, pivots=r.stats.iterations, device_ms=ms,
                       us_per_pivot=ms * 1e3 / max(r.stats.iterations, 1),
                       same_x_bytes=r.x.tobytes() == base.x.tobytes(), same_y_bytes=r.y.tobytes() == base.y.tobytes())
            res["cluster_vs_cta"].append(row)
            print(json.dumps(row), flush=True)
    res["barrier_styles"] = "one built: cluster.sync (release/acquire); the relaxed-arrive and st.async variants not built"
    print(json.dumps({"gpu": res["gpu"], "largest_cluster": largest}))
    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
