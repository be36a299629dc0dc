"""A/B of two builds of the library on the dense simplex paths, in one process tree on one GPU: the build in this tree
("new") against a build of another revision ("old", selected through ELP_LIB_PATH).  The builds alternate, REPS runs
each; every run is a fresh process that solves every case once to warm up and once timed.

Cases (seeded inputs of tests/test_gpu_cluster_simplex.py):
  lp_*        solve_lp, ELP_METHOD_SIMPLEX: mixed(m, n, s) at 40 x 100, 60 x 150, 90 x 120 (12 seeds each), planted 100 x 150
  batch_*     a device-resident batch (elp_batch_run) of 20 000 LPs at 40 x 100 and at 33 x 10 (200 mixed LPs, tiled)
  mip_*       solve_mip: assignment(12, s) (24 x 144) and random_milp(40, 100, s)
  ranging     sensitivity on random_ranging_lp(s, 40, 100)
  cluster_*   transport 60 x 800 and planted 150 x 400 (thread-block clusters in both builds)
  band        planted and mixed LPs at 100 x 170: one CTA in the old build, a 2-CTA cluster in the new one

Every output of a case (status, objective, x, y, pivots, MILP nodes, ranging arrays) is compared byte for byte between
the builds; for `band` the objective is compared to 1e-12 relative instead.  Times: stats.solve_ms (device events) summed
over a case's solves, wall time for ranging; the summary gives per build the median, the spread ((max - min) / median)
and µs per pivot.

    python scripts/gpu_simplex_ab.py --base-lib SO [--reps 5] [--out FILE.jsonl]
    python scripts/gpu_simplex_ab.py --base-src DIR | --base-rev REV      (built into a temp dir, see gpu_stream_ab.py)"""
import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "scripts"))

BAND = "band"           # the one case whose objective may differ in the last bits (one CTA against two)


def cases():
    import test_gpu_cluster_simplex as T
    out = {}
    for m, n in [(40, 100), (60, 150), (90, 120)]:
        out[f"lp_mixed_{m}x{n}"] = ("lp", [T.mixed(m, n, 1000 * m + s) for s in range(12)])
    out["lp_planted_100x150"] = ("lp", [T.planted(100, 150, 7)])
    for m, n in [(40, 100), (33, 10)]:
        out[f"batch_{m}x{n}"] = ("batch", [T.mixed(m, n, 7 * m + s) for s in range(200)])
    out["mip_assignment_12"] = ("mip", [T.assignment(12, s) for s in range(4)])
    out["mip_random_40x100"] = ("mip", [T.random_milp(40, 100, s) for s in range(3)])
    out["ranging_40x100"] = ("ranging", [T.random_ranging_lp(s, m=40, n=100) for s in range(6)])
    out["cluster_transport_60x800"] = ("lp", [T.transport_20x40()])
    out["cluster_planted_150x400"] = ("lp", [T.planted(150, 400, 1)])
    out[BAND] = ("lp", [T.planted(100, 170, 7)] + [T.mixed(100, 170, s) for s in range(4)])
    return out


def run_case(L, kind, ps):
    """solves every problem of a case once; returns (outputs: name -> array, record)"""
    outs, ms, pivots, ctas = {}, 0.0, 0, set()

    def put(k, a):
        outs.setdefault(k, []).append(np.atleast_1d(np.asarray(a)))

    if kind == "lp":
        for p in ps:
            r = L.solve_lp(p["m"], p["n"], p["row_ptr"], p["col_idx"], p["vals"], p["sense"], p["rhs"], p["c"], p["lb"],
                           p["ub"], maximize=p["maximize"], options=L.default_options(method=L.METHOD_SIMPLEX))
            put("status", np.int32(r.status)); put("obj", r.objval); put("x", r.x); put("y", r.y)
            put("pivots", np.int32(r.stats.iterations))
            ms += r.stats.solve_ms; pivots += r.stats.iterations; ctas.add(r.stats.simplex_ctas)
    elif kind == "batch":
        reps = 20000 // len(ps)
        A = np.tile(np.stack([p["A"] for p in ps]), (reps, 1, 1)); b = np.tile(np.stack([p["rhs"] for p in ps]), (reps, 1))
        c = np.stack([np.where(p["maximize"], -p["c"], p["c"]) for p in ps])
        c = np.tile(c, (reps, 1)); lb = np.tile(np.stack([p["lb"] for p in ps]), (reps, 1))
        ub = np.tile(np.stack([p["ub"] for p in ps]), (reps, 1)); sense = np.tile(np.stack([p["sense"] for p in ps]), (reps, 1))
        bt = L.Batch(A, b, c, lb, ub, sense)
        try:
            st = bt.run()
            s, o, x = bt.fetch()
        finally:
            bt.close()
        put("status", s); put("obj", o); put("x", x)
        ms, pivots, ctas = st.solve_ms, st.iterations, {st.simplex_ctas}
    elif kind == "mip":
        for p in ps:
            r = L.solve_mip(p["m"], p["n"], p["row_ptr"], p["col_idx"], p["vals"], p["sense"], p["rhs"], p["c"], p["lb"],
                            p["ub"], p["is_integer"], maximize=p["maximize"], options=L.default_options(max_iter=20000))
            put("status", np.int32(r.status)); put("obj", r.objval); put("x", r.x)
            put("nodes", np.int32(r.stats.restarts)); put("pivots", np.int32(r.stats.iterations))
            ms += r.stats.solve_ms; pivots += r.stats.iterations; ctas.add(r.stats.simplex_ctas)
    else:
        for p in ps:
            t = time.perf_counter()
            res = L.sensitivity(p["m"], p["n"], p["row_ptr"], p["col_idx"], p["vals"], p["sense"], p["rhs"], p["c"], p["lb"],
                                p["ub"], maximize=True)
            ms += (time.perf_counter() - t) * 1e3
            for k, a in zip(("status", "obj", "x", "obj_from", "obj_till", "rhs_from", "rhs_till", "duals"), res):
                put(k, a)
    outs = {k: np.concatenate(v) for k, v in outs.items()}
    rec = {"ms": ms, "pivots": int(pivots), "us_per_pivot": ms * 1e3 / pivots if pivots else None,
           "ctas": sorted(ctas)}
    return outs, rec


def worker(out_dir):
    from easylp_b200 import _lib as L
    os.environ.pop("ELP_SIMPLEX_CLUSTER", None)
    recs = {}
    for name, (kind, ps) in cases().items():
        run_case(L, kind, ps)                                  # warm-up: module load, first launches, workspaces
        outs, rec = run_case(L, kind, ps)
        np.savez(os.path.join(out_dir, name + ".npz"), **outs)
        recs[name] = rec
    print(json.dumps(recs), flush=True)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[0] if out else None
    except (OSError, subprocess.SubprocessError):
        return None


def compare(old_dir, new_dir, name):
    a, b = np.load(os.path.join(old_dir, name + ".npz")), np.load(os.path.join(new_dir, name + ".npz"))
    same = {}
    for k in a.files:
        if name == BAND and k == "obj":
            o, n = a[k], b[k]
            fin = np.isfinite(o)
            same[k] = bool(np.array_equal(o[~fin], n[~fin]) and
                           np.all(np.abs(n[fin] - o[fin]) <= 1e-12 * np.maximum(1.0, np.abs(o[fin]))))
        else:
            same[k] = a[k].tobytes() == b[k].tobytes()
    return same


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--worker", metavar="DIR", help=argparse.SUPPRESS)
    g = ap.add_mutually_exclusive_group()
    g.add_argument("--base-src")
    g.add_argument("--base-rev")
    g.add_argument("--base-lib")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", help="also write the JSON lines to this file")
    args = ap.parse_args()
    if args.worker:
        return worker(args.worker)
    if not (args.base_src or args.base_rev or args.base_lib):
        ap.error("one of --base-src, --base-rev, --base-lib is required")
    from gpu_stream_ab import build_base
    fout = open(args.out, "w") if args.out else None

    def emit(obj):
        line = json.dumps(obj)
        print(line, flush=True)
        if fout:
            fout.write(line + "\n")

    tmp = tempfile.mkdtemp(prefix="elp_simplex_ab_")
    try:
        old_lib = build_base(args, tmp)
        emit({"card": card(), "reps": args.reps})
        runs = {"old": [], "new": []}
        mismatch = {}
        for r in range(args.reps):
            for which in (("old", "new") if r % 2 == 0 else ("new", "old")):
                env = dict(os.environ)
                env.pop("ELP_SIMPLEX_CLUSTER", None)
                if which == "old":
                    env["ELP_LIB_PATH"] = old_lib
                else:
                    env.pop("ELP_LIB_PATH", None)
                d = os.path.join(tmp, f"{which}_{r}")
                os.makedirs(d)
                out = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", d], env=env, cwd=ROOT,
                                     capture_output=True, text=True)
                if out.returncode != 0:
                    sys.stderr.write(out.stderr[-4000:])
                    raise SystemExit(f"{which} worker exited with {out.returncode}")
                recs = json.loads(out.stdout.strip().splitlines()[-1])
                runs[which].append(recs)
                emit({"build": which, "rep": r, "cases": recs})
            for name in runs["new"][-1]:
                same = compare(os.path.join(tmp, f"old_{r}"), os.path.join(tmp, f"new_{r}"), name)
                if not all(same.values()):
                    mismatch.setdefault(name, []).append({"rep": r, "same": same})
        for name in runs["new"][0]:
            summ = {"case": name, "identical": name not in mismatch}
            if name in mismatch:
                summ["mismatch"] = mismatch[name]
            for which in ("old", "new"):
                ms = [x[name]["ms"] for x in runs[which]]
                med = statistics.median(ms)
                upp = [x[name]["us_per_pivot"] for x in runs[which] if x[name]["us_per_pivot"] is not None]
                summ[which] = {"ms": ms, "median_ms": med, "spread": (max(ms) - min(ms)) / med if med else None,
                               "min_ms": min(ms), "max_ms": max(ms), "pivots": sorted({x[name]["pivots"] for x in runs[which]}),
                               "us_per_pivot": statistics.median(upp) if upp else None,
                               "ctas": runs[which][0][name]["ctas"]}
            summ["new_over_old"] = summ["new"]["median_ms"] / summ["old"]["median_ms"] - 1.0
            summ["new_median_within_old_range"] = summ["old"]["min_ms"] <= summ["new"]["median_ms"] <= summ["old"]["max_ms"]
            emit({"summary": summ})
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
        if fout:
            fout.close()


if __name__ == "__main__":
    main()
