#!/usr/bin/env python
"""bench.py — the driver's measurement contract for the EasyLP B200 solve path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload pdlp|batch|transport|mcnf]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

BASELINE.json's metric is compound: "batched LPs/sec; large-LP PDLP iter/s & time-to-1e-6 gap".  The JSON
line's primary `metric` is the large-LP PDLP iteration rate on config 4 (synthetic sparse LP, 2M rows x 4M
cols, ~20M nnz) — the configuration whose SpMV roofline north_star sets the target on.  One step = one
complete solve from the initial iterate to the 1e-6 relative KKT tolerance, so `ms_per_step` IS the
time-to-1e-6-gap.  The batched-simplex number (config 3: 200k dense 20x30 LPs) rides in the same line under
`"batch"` with its own value / e2e / roofline / cpu_baseline; `--workload batch` makes it the primary.
At N = 1 two more sub-lines ride along: `"assembly"` (device CSR assembly of a 21 M-term stream of config 4's matrix,
checked bit-exact) and `"lowering"` (config 2 built through for/sum_for: per-atom evaluation vs one trace + device
expansion, both checked bit-exact).  `--workload mcnf|transport` make configs 5 / 2 the timed PDLP workload.

Timing: device time comes from CUDA events recorded by the library on the stream its kernels run on
(elp_stats.solve_ms); under torchrun the MAX over ranks is taken.  Inputs (2 x 240 MB of matrix per
iteration; 1.1 GB of tableaux per batch) exceed the 126 MB L2, so no flush is needed between steps.
`e2e` goes through the C-ABI call a user of the R package triggers (`$solve()` -> elp_pdlp_create/run/
solution, i.e. what elp_solve_lp does), with pinned HOST buffers, H2D + setup + D2H inside the timed region.

The oracle (oracle/) is loaded ONLY for the `cpu_baseline` leg and `--impl reference`.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it measures (which may be read-only)

from oracle import gen  # noqa: E402  (seeded input generators; not a solve path)
from easylp_b200.partition import lp_ranges, row_block  # noqa: E402


# ------------------------------------------------------------------------------------------------
def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for ln in self.lines:
            f = [s.strip() for s in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(pw)),
                "samples": len(sm), "reasons": sorted(reasons)}


def pinned(a):
    """Copy of `a` in page-locked host memory (torch's pinned allocator; plumbing only)."""
    import torch
    t = torch.from_numpy(np.ascontiguousarray(a))
    try:
        return t.pin_memory().numpy()
    except Exception:
        return t.numpy()


def ncu_traffic(key):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of the dominant kernel, from the committed ncu
    capture of this same workload (profiles/r2_ncu_traffic.json, else round 1's); None when no capture is on file."""
    for name in ("r2_ncu_traffic.json", "r1_ncu_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                t = json.load(f)
            for k in (key + "_gather", key):          # the latest capture of the gather kernels, else the first one
                if k in t:
                    return int(t[k]["dram_bytes"])
        except (OSError, KeyError, ValueError):
            pass
    return None


def pdlp_bytes(m, n, nnz):
    """Algorithmic HBM bytes (DESIGN.md §Kernels; SURVEY §8d): per kernel launch and per iteration."""
    csc = 12 * nnz + 4 * (n + 1) + 8 * m + 56 * n    # A'y SpMV (vals+idx+ptr+y gather) + x,c,l,u,x0 read, x,xbar written
    csr = 12 * nnz + 4 * (m + 1) + 8 * n + 40 * m    # A xbar SpMV + y,lc,uc,y0 read, y written
    return csc, csr, csc + csr


class Dist:
    def __init__(self, want):
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.td = None
        if self.world > 1:
            import torch
            import torch.distributed as td
            torch.cuda.set_device(self.local)
            td.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.td = td
            self.torch = torch
        elif want > 1:
            raise SystemExit(f"--gpus {want} needs torchrun (one process per GPU); see the module docstring")

    def barrier(self):
        if self.td:
            self.td.barrier()
            self.torch.cuda.synchronize()

    def vmax(self, v):
        if not self.td:
            return v
        t = self.torch.tensor([v], dtype=self.torch.float64, device="cuda")
        self.td.all_reduce(t, op=self.td.ReduceOp.MAX)
        return float(t.item())

    def vsum(self, v):
        if not self.td:
            return v
        t = self.torch.tensor([v], dtype=self.torch.float64, device="cuda")
        self.td.all_reduce(t, op=self.td.ReduceOp.SUM)
        return float(t.item())

    def bcast_obj(self, o):
        if not self.td:
            return o
        box = [o]
        self.td.broadcast_object_list(box, src=0)
        return box[0]

    # CPU-side hand-off through the rendezvous store: a rank that waits in an NCCL barrier keeps a spinning kernel on its
    # GPU, which must be idle while rank 0 drives ALL GPUs from one process (e2e_single_call)
    def cpu_signal(self, key):
        if self.td:
            self.td.distributed_c10d._get_default_store().set(key, "1")

    def cpu_wait(self, key):
        if self.td:
            import datetime
            self.td.distributed_c10d._get_default_store().wait([key], datetime.timedelta(minutes=30))

    def close(self):
        if self.td:
            self.td.barrier()
            self.td.destroy_process_group()



PARITY_TOL = 1e-6      # north_star: objective within 1e-6 relative, primal / dual residuals <= 1e-6 relative


def check_parity(L, st, obj, planted, args):
    """status / objective / residual parity of one finished solve; the caller exits non-zero when `ok` is False"""
    out = {"status": L.status_string(st.status), "objective": obj, "planted_objective": planted,
           "rel_primal_res": st.rel_primal_res, "rel_dual_res": st.rel_dual_res, "rel_gap": st.rel_gap, "tol": PARITY_TOL}
    ok = st.status == L.STATUS_OPTIMAL and st.rel_primal_res <= PARITY_TOL and st.rel_dual_res <= PARITY_TOL \
        and st.rel_gap <= PARITY_TOL
    if planted is not None:
        out["objective_rel_err"] = abs(obj - planted) / max(1.0, abs(planted))
        ok = ok and out["objective_rel_err"] <= PARITY_TOL
    out["ok"] = bool(ok)
    return out


def e2e_single_call(args, dist, L, p, steps):
    """N > 1: what an R user gets — ONE process, ONE blocking elp_solve_lp(devices = N) on host buffers.  Rank 0 makes the
    call (worker threads inside the library drive the N GPUs); the other ranks have released their GPUs and wait."""
    N = dist.world
    out = {}
    dist.barrier()
    if dist.rank == 0:
        keys = ("row_ptr", "col_idx", "vals", "sense", "rhs", "c", "lb", "ub")
        hp = {k: pinned(p[k]) for k in keys}
        opt = L.default_options(method=L.METHOD_PDLP, eps_rel=1e-6, max_iter=args.max_iter, devices=N)
        L.set_device(0)

        def call():
            return L.solve_lp(p["m"], p["n"], hp["row_ptr"], hp["col_idx"], hp["vals"], hp["sense"], hp["rhs"], hp["c"],
                              hp["lb"], hp["ub"], maximize=p["maximize"], options=opt)
        r = call()                      # warm-up: worker threads + in-process communicator (kept by the library)
        t0 = time.perf_counter()
        iters = h2d = d2h = 0
        for _ in range(steps):
            r = call()
            iters += r.stats.iterations
            h2d += r.stats.h2d_bytes
            d2h += r.stats.d2h_bytes + 8 * (p["n"] + p["m"])
        dt = time.perf_counter() - t0
        L.release_workspace()
        L.set_device(dist.local)
        out = {"value": iters / dt, "unit": "iter/s", "h2d_bytes_per_step": int(h2d / steps), "d2h_bytes_per_step": int(d2h / steps),
               "s_per_solve": dt / steps, "steps": steps,
               "breakdown": {"setup_s": round(r.stats.setup_ms * 1e-3, 4), "run_device_s": round(r.stats.solve_ms * 1e-3, 4)},
               "path": f"elp_solve_lp(host CSR, devices={N}): one process, one blocking call, {N} worker threads",
               "_stats": r.stats, "_obj": r.objval}
        dist.cpu_signal(f"e2e_done_{p['m']}_{p['n']}")
    else:
        dist.cpu_wait(f"e2e_done_{p['m']}_{p['n']}")        # on the host: this rank's GPU stays idle for rank 0's workers
    dist.barrier()
    return out

# ------------------------------------------------------------------------------------------------
def cpu_pdlp_baseline(p, max_iter, threads):
    from oracle import cbind
    st, out, _, _ = cbind.pdlp(p, eps=1e-6, max_iter=max_iter, nthreads=threads)
    iters, loop_s, setup_s = int(out[1]), float(out[6]), float(out[7])
    return {"value": iters / loop_s, "unit": "iter/s", "cores": threads, "kind": "port",
            "sample": f"first {iters} PDHG iterations of the same LP with oracle/pdlp_ref.c (C + OpenMP r2HPDHG "
                      f"restatement; the reference's lp_solve is not in the image), loop {loop_s:.1f} s + setup {setup_s:.1f} s"}


def cpu_batch_baseline(d, sample, threads):
    from oracle import cbind
    s = slice(0, sample)
    t0 = time.perf_counter()
    cbind.simplex_batch(d["A"][s], d["b"][s], d["c"][s], d["lb"][s], d["ub"][s], d["sense"][s], nthreads=threads)
    dt = time.perf_counter() - t0
    return {"value": sample / dt, "unit": "LP/s", "cores": threads, "kind": "port",
            "sample": f"first {sample} LPs of the same batch with oracle/simplex_ref.c (C + OpenMP bounded primal "
                      f"simplex restatement; the reference's lp_solve is not in the image), {dt:.1f} s"}


def highs_stand_in(args, gpu_c2_s=None, gpu_c3_lps=None):
    """A REAL CPU simplex solver beside the ports (BASELINE.md 3): HiGHS dual simplex (scipy `highs-ds`), labelled a
    stand-in for lp_solve, which is not in this image.  Wall time to the optimum of config 2 (whole solve) and of the first
    `n` LPs of config 3, one core (HiGHS' simplex is serial).  Time-to-solution, not iter/s."""
    try:
        from scipy.optimize import linprog
        from scipy.sparse import csr_matrix
    except Exception as e:                                  # scipy missing on the box: say so, do not fail the bench
        return {"unavailable": str(e)}
    out = {"solver": "HiGHS dual simplex via scipy.optimize.linprog(method='highs-ds'); stand-in for lp_solve 5.5", "cores": 1}
    p = gen.transport(300, 300, seed=0)
    A = csr_matrix((p["vals"], p["col_idx"], p["row_ptr"]), shape=(p["m"], p["n"]))
    le, ge = p["sense"] == 0, p["sense"] == 1
    from scipy.sparse import vstack
    t0 = time.perf_counter()
    r = linprog(p["c"], A_ub=vstack([A[le], -A[ge]]), b_ub=np.r_[p["rhs"][le], -p["rhs"][ge]], bounds=(0, None), method="highs-ds")
    out["c2_transport_s"] = time.perf_counter() - t0
    out["c2_status"], out["c2_objective"] = int(r.status), float(r.fun)
    if gpu_c2_s:
        out["c2_gpu_s"] = gpu_c2_s
        out["c2_speedup_time_to_solution"] = out["c2_transport_s"] / gpu_c2_s
    d = gen.dense_batch(B=args.highs_lps, seed=0)
    t0 = time.perf_counter()
    for i in range(d["B"]):
        linprog(d["c"][i], A_ub=d["A"][i], b_ub=d["b"][i], bounds=list(zip(d["lb"][i], d["ub"][i])), method="highs-ds")
    dt = time.perf_counter() - t0
    out["c3_sample_lps"], out["c3_sample_s"], out["c3_lps_per_s"] = d["B"], dt, d["B"] / dt
    out["c3_note"] = "scipy's per-call overhead is inside this figure (the reference's R loop over lpSolveAPI::solve pays a similar one)"
    if gpu_c3_lps:
        out["c3_speedup_throughput"] = gpu_c3_lps / out["c3_lps_per_s"]
    return out


def host_threads():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


# ------------------------------------------------------------------------------------------------
def bench_pdlp(args, dist, L, p, workload_name):
    """Primary arm: PDLP on a large sparse LP, row-partitioned over dist.world GPUs."""
    N = dist.world
    m, n = p["m"], p["n"]
    nnz = int(p["row_ptr"][m])
    if N > 1:
        uid = dist.bcast_obj(L.comm_unique_id() if dist.rank == 0 else None)
        L.comm_init(N, dist.rank, uid)
        q, r0, r1 = row_block(p, dist.rank, N)
    else:
        q = p
    keys = ("row_ptr", "col_idx", "vals", "sense", "rhs", "c", "lb", "ub")
    hp = {k: pinned(q[k]) for k in keys}
    opt = L.default_options(method=L.METHOD_PDLP, eps_rel=1e-6, max_iter=args.max_iter)

    def create():
        return L.Pdlp(q["m"], n, hp["row_ptr"], hp["col_idx"], hp["vals"], hp["sense"], hp["rhs"], hp["c"], hp["lb"],
                      hp["ub"], maximize=p["maximize"], options=opt, dist=N > 1)

    # ---- value: device-resident handle, one step = one solve to 1e-6 -------------------------------
    h = create()
    for _ in range(args.warmup):
        h.reset()
        h.run()
    sampler = ClockSampler(dist.local)
    dist.barrier()
    if dist.rank == 0:
        sampler.start()
    launches = 0
    dev_ms = 0.0
    iters = 0
    last = None
    t0 = time.perf_counter()
    for _ in range(args.steps):
        h.reset()
        st = h.run()
        dev_ms += st.solve_ms
        launches += st.kernel_launches
        iters += st.iterations
        last = st
    dist.barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    clocks = sampler.stop() if dist.rank == 0 else None
    dev_ms = dist.vmax(dev_ms)
    x, y, obj = h.solution()
    scatter = h.transpose() == L.TRANSPOSE_SCATTER
    ms_csr, ms_csc = h.probe_spmv(20)
    ms_primal, ms_dual = h.probe_step(50)
    h.close()

    # ---- parity gate (north_star): status exact, objective <= 1e-6 relative, residuals <= 1e-6 -- the exit code
    # of this script carries it at every N
    parity = check_parity(L, last, obj, p.get("obj_opt"), args)

    # ---- e2e: the user-facing call with host buffers; H2D + setup + solve + D2H timed -------------
    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    if N > 1:
        e2e = e2e_single_call(args, dist, L, p, e2e_steps)
        parity["e2e_call"] = check_parity(L, e2e.pop("_stats"), e2e.pop("_obj"), p.get("obj_opt"), args) if dist.rank == 0 else None
    dist.barrier()
    t0 = time.perf_counter()
    e2e_iters, h2d, d2h = 0, 0, 0
    parts = {"create_s": 0.0, "run_s": 0.0, "solution_s": 0.0, "close_s": 0.0, "run_device_s": 0.0}
    for _ in range(e2e_steps if N == 1 else 0):
        ta = time.perf_counter()
        hh = create()
        tb = time.perf_counter()
        st = hh.run()
        tc = time.perf_counter()
        hh.solution()
        td_ = time.perf_counter()
        e2e_iters += st.iterations
        h2d += st.h2d_bytes
        d2h += st.d2h_bytes + 8 * (n + q["m"])
        launches_e2e = st.kernel_launches
        hh.close()
        te = time.perf_counter()
        for key, v in (("create_s", tb - ta), ("run_s", tc - tb), ("solution_s", td_ - tc), ("close_s", te - td_),
                       ("run_device_s", st.solve_ms * 1e-3)):
            parts[key] += v / e2e_steps
    dist.barrier()
    e2e_s = dist.vmax(time.perf_counter() - t0)
    if N == 1:
        e2e = {"value": e2e_iters / e2e_s, "unit": "iter/s", "h2d_bytes_per_step": int(h2d / e2e_steps),
               "d2h_bytes_per_step": int(d2h / e2e_steps), "s_per_solve": e2e_s / e2e_steps, "steps": e2e_steps,
               "breakdown": {k: round(v, 4) for k, v in parts.items()},
               "path": "elp_pdlp_create(host CSR) -> elp_pdlp_run -> elp_pdlp_solution (= elp_solve_lp)"}

    peak, peak_src = measured_peak()
    # local matrix of this rank for the roofline (N = 1: the whole matrix)
    ml, nnzl = q["m"], int(q["row_ptr"][q["m"]])
    if N == 1:
        b_csc, b_csr, b_iter = pdlp_bytes(ml, n, nnzl)
    else:
        # rank-local work: K1 on a column block (n/N columns, ~nnz/N entries, gathers the whole y),
        # K2 on the row block (gathers the whole x-bar)
        ncl, nnzc = -(-n // N), nnz // N
        b_csc = 12 * nnzc + 4 * (ncl + 1) + 8 * m + 56 * ncl
        b_csr = 12 * nnzl + 4 * (ml + 1) + 8 * n + 40 * ml
        b_iter = b_csc + b_csr
    b_two_spmv = b_iter                  # SURVEY §8d: what an iteration built from two SpMVs must move
    name_primal = "spmv_warp_kernel<L,NSTW,PrimalEpi> (CSC A'y + fused primal update)"
    name_dual = "spmv_warp_kernel<L,NSTW,DualEpi> (CSR A.xbar + fused dual update)"
    key_primal, key_dual = "primal", "dual"
    if scatter:
        # scatter formulation (single GPU): ONE matrix stream per iteration.  The dual kernel reads the CSR stream, gathers
        # x-bar, updates y and sends val*y_new into g (fp64 reductions resolved in L2: g costs its 8n-byte write-back
        # at most, counted with the primal pass that reads and clears it); the primal pass is elementwise:
        # g, x, c, l, u, x0 read, x-bar, x, g written.
        b_csr = 12 * nnzl + 4 * (ml + 1) + 8 * n + 40 * ml
        b_csc = 72 * n
        b_iter = b_csr + b_csc
        name_primal = "k_primal_from_g (gather-free primal update; reads and clears g = A'y)"
        name_dual = "spmv_warp_kernel<L,NSTW,DualEpi<scatter>> (CSR A.xbar + dual update + RED.ADD.F64 scatter of A'y)"
        key_primal, key_dual = "primal_from_g", "dual_scatter"
    dom_ms, dom_b, dom_name, dom_key = \
        (ms_primal, b_csc, name_primal, key_primal) if ms_primal >= ms_dual else (ms_dual, b_csr, name_dual, key_dual)
    traffic = None
    if N == 1 and args.scale == 1.0:
        traffic = ncu_traffic(dom_key if workload_name.startswith("C4") else workload_name[:2].lower() + "_" + dom_key)
    ach = dom_b / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else 0.0
    iter_ms = dev_ms / max(iters, 1)
    res = {
        "metric": "pdlp_iter_per_s", "value": iters / (dev_ms * 1e-3), "unit": "iter/s", "n_gpus": N,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name, "m": m, "n": n, "nnz": nnz, "eps_rel": 1e-6,
                   "step": "one complete PDLP solve to 1e-6 relative KKT (ms_per_step = time-to-1e-6-gap)",
                   "parallelism": f"row-block x{N}" + (" (K2) + column-block (K1); x-bar / y blocks exchanged by peer stores over NVLink (NCCL all-gather fallback), scalars by NCCL allreduce" if N > 1 else ""),
                   "l2": "matrix (2 x %.0f MB/iter) exceeds the 126 MB L2; no flush needed" % (12 * nnz / 1e6)},
        "time_to_gap_s": dev_ms / args.steps / 1e3,
        "iterations_per_solve": iters / args.steps,
        "status": L.status_string(last.status), "objective": obj, "planted_objective": p.get("obj_opt"),
        "rel_primal_res": last.rel_primal_res, "rel_dual_res": last.rel_dual_res, "rel_gap": last.rel_gap,
        "restarts": last.restarts, "wall_ms_per_step": wall_ms / args.steps,
        "parity": parity,
        "e2e": e2e,
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "kernel": dom_name, "achieved": ach, "peak": peak, "unit": "GB/s",
                     "frac": ach / peak, "frac_of_nominal_8000": ach / 8000.0, "peak_source": peak_src, "traffic": traffic,
                     "bytes_per_launch": dom_b, "ms_per_launch": dom_ms,
                     "formulation": "scatter" if scatter else "gather",
                     "iteration": {"bytes": b_iter, "ms": iter_ms, "achieved": b_iter / (iter_ms * 1e-3) / 1e9,
                                   "frac": b_iter / (iter_ms * 1e-3) / 1e9 / peak,
                                   "two_spmv_bytes": b_two_spmv,
                                   "two_spmv_equivalent_gbs": b_two_spmv / (iter_ms * 1e-3) / 1e9,
                                   "two_spmv_equivalent_frac": b_two_spmv / (iter_ms * 1e-3) / 1e9 / peak,
                                   "note": "whole-solve average incl. check iterations, per rank's local block; "
                                           "`bytes` = what THIS formulation must move, `two_spmv_*` = SURVEY 8d's "
                                           "A.x + A'.y iteration bytes over the same time (equal for 'gather')"},
                     "fused_primal_ms": ms_primal, "fused_dual_ms": ms_dual,
                     "kernel_timing": "CUDA events between the launches of 50 consecutive iterations from a mid-solve iterate",
                     "bare_spmv": {"csr_ms": ms_csr, "csc_ms": ms_csc,
                                   "csr_gbs": (12 * nnzl + 4 * (ml + 1) + 8 * n + 8 * ml) / (ms_csr * 1e-3) / 1e9,
                                   "csc_gbs": (12 * nnzl + 4 * (n + 1) + 8 * ml + 8 * n) / (ms_csc * 1e-3) / 1e9}},
        "clocks": clocks,
        "_outputs": {"x": x, "y": y, "objective": np.array([obj])},
    }
    if N > 1:
        L.comm_destroy()
    return res


def bench_batch(args, dist, L, d):
    """Batched dense simplex; LPs sharded contiguously over ranks, no collective."""
    N = dist.world
    B, m, n = d["B"], d["m"], d["n"]
    lo, hi = lp_ranges(B, N)[dist.rank]
    keys = ("A", "b", "c", "lb", "ub", "sense")
    hp = {k: pinned(d[k][lo:hi]) for k in keys}
    Bl = hi - lo
    h = L.Batch(hp["A"], hp["b"], hp["c"], hp["lb"], hp["ub"], hp["sense"])
    for _ in range(args.warmup):
        h.run()
    sampler = ClockSampler(dist.local)
    dist.barrier()
    if dist.rank == 0:
        sampler.start()
    dev_ms, launches = 0.0, 0
    for _ in range(args.steps):
        st = h.run()
        dev_ms += st.solve_ms
        launches += st.kernel_launches
    dist.barrier()
    clocks = sampler.stop() if dist.rank == 0 else None
    dev_ms = dist.vmax(dev_ms)
    status, obj, x = h.fetch()
    h.close()
    n_opt = dist.vsum(float((status == 0).sum()))
    # e2e through elp_solve_batch with host buffers
    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    out = (pinned(np.zeros(Bl, np.int32)), pinned(np.zeros(Bl)), pinned(np.zeros((Bl, n))))
    L.solve_batch(hp["A"], hp["b"], hp["c"], hp["lb"], hp["ub"], hp["sense"], out=out)      # warm-up: workspace + streams
    dist.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        s2, o2, x2, st2 = L.solve_batch(hp["A"], hp["b"], hp["c"], hp["lb"], hp["ub"], hp["sense"], out=out)
    dist.barrier()
    e2e_s = dist.vmax(time.perf_counter() - t0)
    assert np.array_equal(s2, status) and np.array_equal(o2, obj), "streamed elp_solve_batch differs from the resident batch"
    pivots = dist.vsum(float(st2.iterations))
    peak, peak_src = measured_peak()
    bytes_lp = 8 * (m * n + m + 3 * n) + m + 8 * (n + 1) + 4 + 4
    ms = dev_ms / args.steps
    ach = bytes_lp * Bl / (ms * 1e-3) / 1e9
    return {
        "metric": "batched_lps_per_s", "value": B * args.steps / (dev_ms * 1e-3), "unit": "LP/s", "n_gpus": N,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"C3: batch of {B} random feasible dense LPs ({m} constraints x {n} vars), batched simplex",
                   "parallelism": f"LP ranges x{N}, no collective",
                   "l2": "batch data (%.2f GB) exceeds the 126 MB L2; no flush needed" % (bytes_lp * B / 1e9)},
        "optimal": int(n_opt), "pivots_per_lp": pivots / B, "pivots_per_s": pivots / ms * 1e3,
        "parity": {"ok": bool(int(n_opt) == B), "optimal": int(n_opt), "of": B,
                   "note": "every LP of the batch is feasible and bounded by construction: status must be optimal for all"},
        "e2e": {"value": B * e2e_steps / e2e_s, "unit": "LP/s", "h2d_bytes_per_step": int(st2.h2d_bytes * N),
                "d2h_bytes_per_step": int(st2.d2h_bytes * N), "path": "elp_solve_batch(host arrays)"},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "kernel": "simplex_warp_kernel<MR,CPL> (one LP per warp, tableau in shared memory)", "achieved": ach, "peak": peak, "unit": "GB/s",
                     "frac": ach / peak, "peak_source": peak_src,
                     "traffic": ncu_traffic("batch") if (dist.world == 1 and B == 200_000 and m == 20 and n == 30) else None,
                     "bytes_per_launch": bytes_lp * Bl,
                     "ms_per_launch": ms,
                     "note": "HBM fraction is the mandated figure; shared-memory bandwidth and instruction issue of the pivot chain bound this kernel (ncu: LSU wavefronts 76 %, issue 56 %)"},
        "clocks": clocks,
        "_outputs": {"status": status, "objective": obj, "x": x},
    }


def bench_assembly(args, L, p):
    """Kernel (1): device CSR assembly of the workload's own matrix handed over as an emission-order term list
    (oracle/gen.py::term_stream: seeded permutation + 5 % split duplicates).  Checked bit-exact on the spot."""
    m, n = p["m"], p["n"]
    nnz = int(p["row_ptr"][m])
    r, c, v = gen.term_stream(p, 0.05, 0)
    hr, hc, hv = pinned(r), pinned(c), pinned(v)
    T = int(r.size)
    dev_ms, tot_ms = [], []
    for i in range(args.warmup + args.steps):
        rp, ci, vv, st = L.assemble_csr(hr, hc, hv, m, n)
        if i >= args.warmup:
            dev_ms.append(st.solve_ms)
            tot_ms.append(st.total_ms)
    exact = bool(np.array_equal(rp, p["row_ptr"]) and np.array_equal(ci, p["col_idx"]) and vv.tobytes() == p["vals"].tobytes())
    # the same terms in the order `$con()` emits them (row after row, columns ascending): detected on the device, no sort
    order = np.lexsort((c, r))
    sr, sc, sv = pinned(r[order]), pinned(c[order]), pinned(v[order])
    s_ms = []
    for i in range(args.warmup + args.steps):
        rp2, ci2, vv2, st2 = L.assemble_csr(sr, sc, sv, m, n)
        if i >= args.warmup:
            s_ms.append(st2.solve_ms)
    exact = exact and bool(np.array_equal(rp2, p["row_ptr"]) and np.array_equal(ci2, p["col_idx"]) and vv2.tobytes() == p["vals"].tobytes())
    peak, peak_src = measured_peak()
    alg_of = lambda T_, nnz_, m_: 16 * T_ + 12 * nnz_ + 4 * (m_ + 1)      # noqa: E731  (SURVEY 8d)
    alg = alg_of(T, nnz, m)
    ms = float(np.mean(dev_ms))
    return {"metric": "assembly_terms_per_s", "value": T / (ms * 1e-3), "unit": "terms/s", "terms": T, "nnz": nnz,
            "bit_exact": exact, "ms_per_step": ms,
            "e2e": {"value": T / (float(np.mean(tot_ms)) * 1e-3), "unit": "terms/s", "h2d_bytes_per_step": 16 * T,
                    "d2h_bytes_per_step": 12 * nnz + 4 * (m + 1), "path": "elp_assemble_csr(host term list)"},
            "gpu_launches": int(st.kernel_launches),
            "ordered_stream": {"ms_per_step": float(np.mean(s_ms)), "terms_per_s": T / (float(np.mean(s_ms)) * 1e-3),
                               "achieved_gbs": alg_of(T, nnz, m) / (float(np.mean(s_ms)) * 1e-3) / 1e9,
                               "frac": alg_of(T, nnz, m) / (float(np.mean(s_ms)) * 1e-3) / 1e9 / peak,
                               "gpu_launches": int(st2.kernel_launches),
                               "traffic": ncu_traffic("assembly_ordered") if args.scale == 1.0 else None,
                               "note": "same terms in `$con()` emission order (rows ascending, columns ascending): two passes "
                                       "straight over the stream (order + counts, fold + emit), no keys, no sort"},
            "roofline": {"bound": "hbm",
                         "kernel": ("row-bucket split + shared-memory sort-and-fold per bucket + emit (bucket_sort.cuh)"
                                    if st.kernel_launches < 20 else "radix sort passes + ordered fold + scan + scatter")
                                   + f" ({int(st.kernel_launches)} launches)",
                         "achieved": alg / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": alg / (ms * 1e-3) / 1e9 / peak, "peak_source": peak_src,
                         "traffic": ncu_traffic("assembly") if (st.kernel_launches < 20 and args.scale == 1.0) else None,
                         "bytes_per_launch": alg, "ms_per_launch": ms,
                         "note": "algorithmic bytes 16 T + 12 nnz + 4 (m+1) over the whole assembly, unordered stream; "
                                 "round 1 sorted with 6 LSD passes (~8x the algorithmic bytes, 3.4 ms); the bucket path "
                                 "moves ~100 B per term"}}


def bench_lowering(args, L):
    """SURVEY 8f N2: BASELINE config 2 (transport 300 x 300) written with for + sum_for.  `eager` evaluates the body once
    per atom / grid row on the host (the reference's interpreter loop, R/utils.R:50-53,405-408) and ships 180 000 terms;
    `lowered` traces each body once and lets the device expand the index-set families (elp_assemble_lowered).  Both
    must give the generator's canonical CSR bit for bit."""
    from easylp_b200 import model as M
    S = T = 300
    p = gen.transport(S, T, seed=0)
    src, snk = list(range(1, S + 1)), list(range(1, T + 1))

    def build(lowering):
        M.LOWERING = lowering
        try:
            t0 = time.perf_counter()
            lp = M.easylp()
            x = lp.var("x", src, snk, lower=0)
            cost = M.parameter(p["cost"].ravel(order="F"), src, snk)
            supply, demand = M.parameter(p["supply"], src), M.parameter(p["demand"], snk)
            lp.min(M.sum_for(lambda s, t: cost[s, t] * x[s, t], s=src, t=snk))
            lp.con(make=M.for_(lambda s: M.sum_for(lambda t: x[s, t], t=snk) <= supply[s], s=src),
                   sell=M.for_(lambda t: M.sum_for(lambda s: x[s, t], s=src) >= demand[t], t=snk))
            t1 = time.perf_counter()
            rp, ci, v = lp._csr()
            c = lp.objective_fun
            t2 = time.perf_counter()
        finally:
            M.LOWERING = True
        exact = bool(np.array_equal(rp, p["row_ptr"]) and np.array_equal(ci, p["col_idx"])
                     and np.asarray(v).tobytes() == p["vals"].tobytes() and c.tobytes() == p["c"].tobytes()
                     and lp.constraint.rhs.tobytes() == p["rhs"].tobytes())
        st = lp.assembly_stats
        return dict(host_s=t1 - t0, assemble_s=t2 - t1, total_s=t2 - t0, device_ms=st.solve_ms, bit_exact=exact,
                    h2d_bytes=int(st.h2d_bytes), gpu_launches=int(st.kernel_launches))

    build(True)                                     # warm-up (workspace, module load)
    low = build(True)
    eag = build(False)
    return {"metric": "model_build_s", "unit": "s", "higher_is_better": False,
            "workload": "C2: transport 300 x 300 (90 000 vars, 600 rows, 180 000 nnz) through for_/sum_for, objective via sum_for",
            "value": low["total_s"], "lowered": low, "eager": eag, "speedup": eag["total_s"] / low["total_s"],
            "gpu_launches": low["gpu_launches"]}


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Writes each array as out_dir/<name>.npy in float64, so that two builds can be compared output for output.  When the
    arrays exceed DUMP_BYTES in all, each is cut to its share of the budget: a seeded sample of its flattened elements,
    the same indices on every run with the same arguments."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.asarray(v, np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > DUMP_BYTES:
            keep = a.size * DUMP_BYTES // total
            a = a.ravel()[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------
def golden_objective(key):
    try:
        with open(os.path.join(ROOT, "tests", "golden", "configs.json")) as f:
            return float.fromhex(json.load(f)[key]["objective"])
    except (OSError, KeyError, ValueError):
        return None


def make_problem(args):
    w = args.workload
    if w == "pdlp":
        m = int(round(2_000_000 * args.scale))
        return gen.sparse_planted(m, seed=0), f"C4: synthetic sparse LP {m} rows x {2 * m} cols, planted optimum, PDLP to 1e-6"
    if w == "transport":
        p = gen.transport(300, 300, seed=0)
        p["obj_opt"] = golden_objective("c2_transport_300x300_seed0")     # HiGHS (tests/golden/make_configs.py)
        return p, "C2: transportation 300 x 300 (90k vars, 600 rows), PDLP to 1e-6"
    if w == "mcnf":
        K = max(1, int(round(50 * args.scale)))
        p = gen.mcnf(K=K)
        if K == 50:
            p["obj_opt"] = golden_objective("c5_mcnf_K50_seed0")          # shortest-path decomposition, capacities slack
        return p, f"C5: multi-commodity flow, {K} commodities on 20k nodes / 100k arcs, PDLP to 1e-6"
    raise SystemExit(f"unknown workload {w}")


def run_reference(args):
    """--impl reference: the CPU restatement of the path on the host cores, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = host_threads()
    if args.workload == "batch":
        d = gen.dense_batch(B=int(200_000 * args.scale), seed=0)
        sample = min(d["B"], args.cpu_sample_lps)
        vals = []
        for i in range(args.warmup + args.steps):
            r = cpu_batch_baseline(d, sample, threads)
            if i >= args.warmup:
                vals.append(r["value"])
        v = float(np.mean(vals))
        line = {"metric": "batched_lps_per_s", "value": v, "unit": "LP/s", "ms_per_step": sample / v * 1e3,
                "config": {"workload": f"C3: batch of {d['B']} dense LPs (20 x 30); each step = first {sample} LPs"}}
        base = r
    else:
        p, name = make_problem(args)
        vals = []
        for i in range(args.warmup + args.steps):
            r = cpu_pdlp_baseline(p, args.cpu_sample_iters, threads)
            if i >= args.warmup:
                vals.append(r["value"])
        v = float(np.mean(vals))
        line = {"metric": "pdlp_iter_per_s", "value": v, "unit": "iter/s", "ms_per_step": args.cpu_sample_iters / v * 1e3,
                "config": {"workload": name + f"; each step = first {args.cpu_sample_iters} iterations"}}
        base = r
    base = dict(base)
    base["value"] = v
    line.update({"impl": "reference",
                 "reference_is": "CPU PORT of this repo's own algorithm (oracle/, C + OpenMP, all host threads) — NOT lp_solve: "
                                 "R and lpSolveAPI are not in the image, and the reference's dense DSL cannot even build "
                                 "configs 2-5 (SURVEY 0.3).  A real CPU solver (HiGHS dual simplex, stand-in) is timed in the "
                                 "main arm's cpu_baseline.alt.",
                 "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                 "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                 "cpu_baseline": base, "gpu_launches": 0,
                 "e2e": {"value": v, "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="pdlp", choices=["pdlp", "batch", "transport", "mcnf"])
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the workload (smoke runs only; 1.0 = BASELINE size)")
    ap.add_argument("--max-iter", type=int, default=400_000)
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--cpu-sample-iters", type=int, default=150)
    ap.add_argument("--cpu-sample-lps", type=int, default=20_000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--highs-lps", type=int, default=2000, help="LPs of config 3 given to the HiGHS stand-in")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary (batch) arm in the pdlp line")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the primary arm's last timed step returned (x, y, objective of the PDLP solve; "
                         "status, objective, x of the batch) as DIR/<name>.npy, float64, at most 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    if args.impl == "reference":
        run_reference(args)
        return

    dist = Dist(args.gpus)
    from easylp_b200 import _lib as L
    if L.device_count() < 1:
        raise SystemExit("bench.py needs a CUDA device: libeasylp_b200 has no CPU fallback")
    L.set_device(dist.local)
    threads = host_threads()

    if args.workload == "batch":
        d = gen.dense_batch(B=int(200_000 * args.scale), seed=0)
        res = bench_batch(args, dist, L, d)
        outputs = res.pop("_outputs")
        if dist.rank == 0 and dist.world == 1 and not args.no_cpu_baseline:
            res["cpu_baseline"] = cpu_batch_baseline(d, min(d["B"], args.cpu_sample_lps), threads)
    else:
        p, name = make_problem(args)
        res = bench_pdlp(args, dist, L, p, name)
        outputs = res.pop("_outputs")
        if not args.no_secondary:
            d = gen.dense_batch(B=int(200_000 * args.scale), seed=0)
            sec = bench_batch(args, dist, L, d)
            if dist.rank == 0 and dist.world == 1 and not args.no_cpu_baseline:
                sec["cpu_baseline"] = cpu_batch_baseline(d, min(d["B"], args.cpu_sample_lps), threads)
            res["batch"] = {k: sec[k] for k in ("metric", "value", "unit", "ms_per_step", "config", "optimal", "parity",
                                                "pivots_per_lp", "pivots_per_s", "e2e", "gpu_launches", "roofline")
                            if k in sec}
            if "cpu_baseline" in sec:
                res["batch"]["cpu_baseline"] = sec["cpu_baseline"]
            res["gpu_launches"] += sec["gpu_launches"]
        if dist.world == 1 and not args.no_secondary:
            asm = bench_assembly(args, L, p)
            res["assembly"] = asm
            res["gpu_launches"] += asm["gpu_launches"] * args.steps
            if dist.rank == 0:
                res["lowering"] = bench_lowering(args, L)
        if dist.world == 1 and not args.no_secondary and args.workload == "pdlp":
            # config 5 rides along: the structured LP where the SpMV kernel passes 60 % of the HBM roofline, with its own
            # roofline block and the independently pinned objective; config 2 gives the time-to-solution the HiGHS
            # stand-in is compared with
            sub_args = argparse.Namespace(**vars(args))
            sub_args.steps, sub_args.warmup, sub_args.e2e_steps = max(3, min(args.steps, 5)), 3, 2
            for key, wl in (("mcnf", "mcnf"), ("transport", "transport")):
                sub_args.workload = wl
                q, qname = make_problem(sub_args)
                sub = bench_pdlp(sub_args, dist, L, q, qname)
                res[key] = {k: sub[k] for k in ("metric", "value", "unit", "ms_per_step", "time_to_gap_s", "iterations_per_solve",
                                                "config", "parity", "e2e", "gpu_launches", "roofline") if k in sub}
                res["gpu_launches"] += sub["gpu_launches"]
        if dist.rank == 0 and dist.world == 1 and not args.no_cpu_baseline:
            res["cpu_baseline"] = cpu_pdlp_baseline(p, args.cpu_sample_iters, threads)
            res["cpu_baseline"]["alt"] = highs_stand_in(args, gpu_c2_s=res.get("transport", {}).get("time_to_gap_s"),
                                                        gpu_c3_lps=res.get("batch", {}).get("e2e", {}).get("value"))
    if dist.rank == 0:
        print(json.dumps(res), flush=True)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
    dist.close()
    # the exit code carries parity: a wrong status / objective / residual at any N is a failed run, not a slow one
    bad = []
    par = res.get("parity")
    if par is not None and not par["ok"]:
        bad.append(f"pdlp parity: {par}")
    if par is not None and par.get("e2e_call") and not par["e2e_call"]["ok"]:
        bad.append(f"pdlp parity of the single-call e2e: {par['e2e_call']}")
    for key in ("batch", "mcnf"):
        sub = res if res.get("metric") == "batched_lps_per_s" and key == "batch" else res.get(key)
        if isinstance(sub, dict) and sub.get("parity") is not None and not sub["parity"]["ok"]:
            bad.append(f"{key} parity: {sub['parity']}")
    for key in ("assembly", "lowering"):
        sub = res.get(key)
        if isinstance(sub, dict):
            exact = sub.get("bit_exact", True) and sub.get("lowered", {}).get("bit_exact", True) and sub.get("eager", {}).get("bit_exact", True)
            if not exact:
                bad.append(f"{key}: CSR not bit-exact")
    if bad:
        print("PARITY FAILURE: " + "; ".join(bad), file=sys.stderr, flush=True)
        sys.exit(3)


if __name__ == "__main__":
    main()
