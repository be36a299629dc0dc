"""A/B of two builds of the library on the PDLP workloads, in one process tree on one GPU: the build in this tree ("new")
against a build of another revision ("old"), selected through ELP_LIB_PATH.  The two builds alternate, REPS runs each,
on pdlp (C4), mcnf (C5) and transport (C2).  Prints one JSON line per run and a summary line per workload: per-run iter/s,
median and spread (max - min over median), the fused kernel times, whether x, y and the objective dumped by
`bench.py --dump-outputs` are byte-identical between the builds, and the iteration and restart counts.

    python scripts/gpu_stream_ab.py --base-src DIR     # DIR: a source tree of the old revision (built here into a temp dir)
    python scripts/gpu_stream_ab.py --base-rev REV     # the same from `git archive REV` (needs a git checkout)
    python scripts/gpu_stream_ab.py --base-lib SO      # an already built old library

The C4 roofline fraction in bench.py counts the bytes of the parent's epilogues (56 B per column, 40 B per row); the
summary also gives the fraction for the bytes the new plain iterations move (`alg_bytes_new`)."""
import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def build_base(args, tmp):
    if args.base_lib:
        return os.path.abspath(args.base_lib)
    src = os.path.join(tmp, "base")
    if args.base_src:
        shutil.copytree(os.path.join(args.base_src, "easylp_b200", "csrc"), os.path.join(src, "easylp_b200", "csrc"))
        shutil.copytree(os.path.join(args.base_src, "include"), os.path.join(src, "include"))
    else:
        os.makedirs(src)
        tar = subprocess.run(["git", "-C", ROOT, "archive", args.base_rev, "easylp_b200/csrc", "include"], check=True,
                             capture_output=True).stdout
        subprocess.run(["tar", "-x", "-C", src], input=tar, check=True)
    subprocess.run(["make", "-s", "-j8", "-C", os.path.join(src, "easylp_b200", "csrc")], check=True)
    return os.path.join(src, "easylp_b200", "libeasylp_b200.so")


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[0] if out else None
    except (OSError, subprocess.SubprocessError):
        return None


def bench(lib, workload, dump, args):
    env = dict(os.environ)
    if lib:
        env["ELP_LIB_PATH"] = lib
    else:
        env.pop("ELP_LIB_PATH", None)
    steps, warmup = (args.steps, args.warmup) if workload == "pdlp" else (args.small_steps, args.warmup)
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup),
           "--workload", workload, "--no-secondary", "--no-cpu-baseline", "--dump-outputs", dump]
    out = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True)
    if out.returncode != 0:
        sys.stderr.write(out.stderr[-4000:])
        raise SystemExit(f"bench.py {workload} exited with {out.returncode}")
    line = [s for s in out.stdout.splitlines() if s.startswith("{")][-1]
    return json.loads(line)


def new_bytes(m, n, nnz, l_streamed, u_streamed, rhs_sense):
    """bytes the plain iterations of this tree move: K1 reads x-bar, c, [l], [u], x0 and writes x-bar; K2 reads y, rhs +
    sense (or lc, uc), y0 and writes y"""
    csc = 12 * nnz + 4 * (n + 1) + 8 * m + (8 * (4 + l_streamed + u_streamed)) * n
    csr = 12 * nnz + 4 * (m + 1) + 8 * n + (33 if rhs_sense else 40) * m
    return csc + csr


def main():
    ap = argparse.ArgumentParser()
    g = ap.add_mutually_exclusive_group(required=True)
    g.add_argument("--base-src")
    g.add_argument("--base-rev")
    g.add_argument("--base-lib")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=1, help="timed solves per C4 run")
    ap.add_argument("--small-steps", type=int, default=3, help="timed solves per C5 / C2 run")
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--workloads", default="pdlp,mcnf,transport")
    args = ap.parse_args()
    tmp = tempfile.mkdtemp(prefix="elp_ab_")
    try:
        old_lib = build_base(args, tmp)
        print(json.dumps({"card": card(), "old_lib": old_lib}), flush=True)
        for wl in args.workloads.split(","):
            runs = {"old": [], "new": []}
            for r in range(args.reps):
                order = ("old", "new") if r % 2 == 0 else ("new", "old")
                for which in order:
                    dump = os.path.join(tmp, f"{wl}_{which}")
                    res = bench(old_lib if which == "old" else None, wl, dump, args)
                    rf = res.get("roofline", {})
                    rec = {"workload": wl, "build": which, "rep": r, "value": res["value"],
                           "iterations_per_solve": res["iterations_per_solve"], "restarts": res["restarts"],
                           "status": res["status"], "objective": res["objective"],
                           "fused_primal_ms": rf.get("fused_primal_ms"), "fused_dual_ms": rf.get("fused_dual_ms"),
                           "iteration_ms": rf.get("iteration", {}).get("ms"), "peak_gbs": rf.get("peak"),
                           "bench_frac": rf.get("iteration", {}).get("frac"), "config": res["config"]}
                    runs[which].append(rec)
                    print(json.dumps({k: v for k, v in rec.items() if k != "config"}), flush=True)
                same = {}
                for name in ("x", "y", "objective"):
                    a = np.load(os.path.join(tmp, f"{wl}_old", name + ".npy"))
                    b = np.load(os.path.join(tmp, f"{wl}_new", name + ".npy"))
                    same[name] = a.tobytes() == b.tobytes()
                print(json.dumps({"workload": wl, "rep": r, "outputs_bit_identical": same}), flush=True)
                if not all(same.values()):
                    runs.setdefault("mismatch", []).append(r)
            summ = {"workload": wl}
            for which in ("old", "new"):
                v = [x["value"] for x in runs[which]]
                med = statistics.median(v)
                summ[which] = {"values": v, "median": med, "spread": (max(v) - min(v)) / med,
                               "fused_primal_ms": statistics.median(x["fused_primal_ms"] for x in runs[which]),
                               "fused_dual_ms": statistics.median(x["fused_dual_ms"] for x in runs[which]),
                               "iterations_per_solve": sorted({x["iterations_per_solve"] for x in runs[which]}),
                               "restarts": sorted({x["restarts"] for x in runs[which]})}
            summ["gain"] = summ["new"]["median"] / summ["old"]["median"] - 1.0
            summ["gain_over_spread"] = summ["gain"] / max(summ["old"]["spread"], summ["new"]["spread"], 1e-12)
            summ["outputs_bit_identical"] = "mismatch" not in runs
            summ["counts_equal"] = (summ["old"]["iterations_per_solve"] == summ["new"]["iterations_per_solve"] and
                                    summ["old"]["restarts"] == summ["new"]["restarts"])
            if wl == "pdlp":
                cfg = runs["new"][0]["config"]
                m, n, nnz = cfg["m"], cfg["n"], cfg["nnz"]
                b = new_bytes(m, n, nnz, 0, 1, True)          # C4: l = 0 (not streamed), u = 1e3 (streamed), rhs + sense
                it_ms = statistics.median(x["iteration_ms"] for x in runs["new"])
                summ["alg_bytes_new"] = b
                summ["frac_new_bytes"] = b / (it_ms * 1e-3) / 1e9 / runs["new"][0]["peak_gbs"]
                summ["bench_frac_parent_bytes"] = statistics.median(x["bench_frac"] for x in runs["new"])
            print(json.dumps({"summary": summ}), flush=True)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
