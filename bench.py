#!/usr/bin/env python
"""bench.py — PDLP iterations/sec on BASELINE.json's headline workload: the synthetic sparse LP with 10M variables x
10M constraints, 8 nnz/row, fp64 (configs[3]'s instance; it fits one B200, so every N = 1, 2, 4, 8 runs the SAME LP and
the N-GPU numbers are strong scaling).  --workload c2 selects configs[1] (1M x 1M), --workload c3 the pds-shaped
multicommodity LP of configs[2] (both single-GPU profile workloads).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (through the C ABI)
  python bench.py --impl reference --gpus N --steps K ...  # CPU arm: the oracle port of the reference PDLP on host cores
  python bench.py ... --dump-outputs DIR                   # also save the last timed step's results as DIR/*.npy

A "step" = one solve of ITERS_PER_STEP PDLP iterations on the resident LP (tolerances 0 => never stops early).
  value  = accepted PDLP iterations / device time of the solver loop (CUDA events, inputs resident in HBM)
  e2e    = the same through cuOptCreateRangedProblem + cuOptSolve + cuOptGet*Solution with HOST buffers:
           H2D upload, transpose, diagonal scaling and D2H of the solution are inside the timed region
Prints ONE JSON line (rank 0).
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
sys.path.insert(0, ROOT)

METRIC = "pdlp_iterations_per_sec"
UNIT = "iterations/s"
ITERS_PER_STEP = 2000


def usable_cores() -> int:
    """Host cores this process may really use: min(cpu_count, affinity mask, cgroup CPU quota).  A container that shows
    128 CPUs but is throttled to a few makes a 128-thread OpenMP run slower than an 8-thread one (measured: 2.1 vs 4.7
    iterations/s on the 10M LP), so the CPU legs size their thread pool with this."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:  # noqa: BLE001
        pass
    for path, parse in (("/sys/fs/cgroup/cpu.max", lambda t: t.split()),
                        ("/sys/fs/cgroup/cpu/cpu.cfs_quota_us", None)):
        try:
            with open(path) as f:
                txt = f.read().strip()
            if parse:
                quota, period = parse(txt)
                if quota != "max":
                    n = min(n, max(1, int(float(quota) / float(period) + 0.5)))
            else:
                with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                    period = float(f.read().strip())
                if float(txt) > 0:
                    n = min(n, max(1, int(float(txt) / period + 0.5)))
        except Exception:  # noqa: BLE001
            pass
    return max(1, min(n, 64))  # beyond ~64 threads the memory-bound CPU SpMV stops scaling


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:  # noqa: BLE001
        return {"hbm_gbs": 6650.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([t.strip() for t in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


WORKLOADS = {"c4": (10_000_000, 10_000_000), "c2": (1_000_000, 1_000_000)}
# dram__bytes_read.sum + dram__bytes_write.sum per step of the dominant kernel (group), from the COMMITTED `ncu --set full`
# captures under profiles/ (bench.py never runs under a profiler): (workload, kernel, blocked) -> (bytes, file).  The line
# says `traffic_source: committed capture` so that nobody mistakes it for an in-run measurement.
NCU_TRAFFIC = {}
try:
    with open(os.path.join(ROOT, "profiles", "r2", "ncu_traffic.json")) as _f:
        for _e in json.load(_f)["entries"]:
            NCU_TRAFFIC[(_e["workload"], _e["kernel"], bool(_e["blocked"]))] = (_e["bytes_per_step"], _e["source"])
except Exception:  # noqa: BLE001
    pass
TRANSPORTS = {"gather": "every rank owns 1/N of the rows of A and 1/N of the rows of A^T; xbar and y' are all-gathered by NVLink "
                        "peer stores issued by the kernels that produce them (K1, K2), 3 scalars per rank; no partial "
                        "products, no NCCL inside the PDHG loop",
              "p2p": "NVLink peer stores issued by the producing kernels (xbar slices, A_g^T y partials, 3 scalars); "
                     "no NCCL inside the PDHG loop",
              "nccl": "NCCL all-gather(xbar) + reduce-scatter(A_g^T y) + all-reduce(3 scalars) per attempt",
              "allreduce": "primal side replicated, one NCCL all-reduce of n+1 doubles per attempt"}


def workload(args):
    from cuopt_b200 import lpgen
    if args.workload == "c3":
        return lpgen.multicommodity(nodes=9000, arcs=27000, commodities=11, seed=1234)
    rows, cols = WORKLOADS[args.workload]
    # --locality rho: fraction of each row's columns drawn from the row's own 1/8 column band (SURVEY §8d, C4's knob;
    # 0 = uniform columns, the worst case for the gathers and the default)
    return lpgen.sparse_lp(args.rows or rows, args.cols or cols, args.nnz_per_row, seed=1234, locality=args.locality)


def config_dict(args, lp, n_gpus):
    names = {"c4": "configs[3] instance (the 10M-var LP the metric is quoted on)", "c2": "configs[1]",
             "c3": "configs[2] (pds-shaped multicommodity flow, synthesised: no pds file in the tree)"}
    transport = os.environ.get("CUOPT_B200_DIST_MODE", "gather")
    return {"workload": f"{names[args.workload]}: {lp.name}, {lp.m}x{lp.n}, nnz {lp.nnz}, fp64",
            "rows": lp.m, "cols": lp.n, "nnz": lp.nnz, "iterations_per_step": args.iters,
            "pdlp_solver_mode": "Stable2",
            "parallelism": (f"ONE LP: constraint rows and primal column slices sharded over {n_gpus} GPUs (one process "
                            f"each); transport: {TRANSPORTS[transport]}") if n_gpus > 1 else "1 GPU",
            "l2_policy": "per-iteration working set (A, A^T, 14 vectors = %.0f MB) exceeds the 126 MB L2"
                         % (lp.algorithmic_bytes_per_iteration() / 1e6)}


def time_cpu_oracle(lp, cores, iterations, repeats):
    """ONE protocol for both CPU numbers of this file (cpu_baseline of the GPU arm, the --impl reference arm): the oracle
    port with `cores` OpenMP threads, initialised, then 12 untimed iterations — the first 10 PDLP iterations are each a
    major iteration (termination evaluation + restart test, pdlp.cu:1082-1090), which is not the steady state the metric
    is about — then `repeats` timed samples of `iterations` iterations.  Returns (iterations/s, seconds per sample)."""
    from oracle import pdlp_oracle as po
    o = po.Oracle(lp.offsets, lp.indices, lp.values, lp.c, lp.var_lb, lp.var_ub, lp.con_lb, lp.con_ub, tol=0.0,
                  num_threads=cores)
    o.initialise()
    o.run(12)
    t0 = time.perf_counter()
    for _ in range(repeats):
        o.run(iterations)
    dt = time.perf_counter() - t0
    return repeats * iterations / dt, dt / repeats


def reference_dual_simplex_leg(lp, cap_seconds):
    """SURVEY 8(d): the reference's OWN CPU path for an LP is its dual simplex (single-threaded, dual_simplex/solve.hpp:64-67),
    compiled unchanged into oracle/_ref.  On the 1M / 10M workloads it is not expected to finish: it runs in a child process
    under `cap_seconds` and the outcome — optimal with its time, or DNF — is reported, never omitted."""
    import multiprocessing as mp

    def child(q):
        try:
            from oracle import ref_cpu
            if not ref_cpu.available():
                q.put({"status": "unavailable", "why": "oracle/_ref/libcuopt_ref_cpu.so not built on this box"})
                return
            r = ref_cpu.dual_simplex(lp.offsets, lp.indices, lp.values, lp.con_lb, lp.con_ub, lp.c, lp.var_lb, lp.var_ub,
                                     time_limit=float(cap_seconds))
            q.put({"status": r["status"], "objective": r["objective"], "iterations": r["iterations"], "seconds": r["seconds"]})
        except Exception as e:  # noqa: BLE001
            q.put({"status": "error", "why": str(e)[:200]})

    ctx = mp.get_context("fork")
    q = ctx.Queue()
    pr = ctx.Process(target=child, args=(q,))
    t0 = time.perf_counter()
    pr.start()
    pr.join(cap_seconds + 60.0)
    out = {"status": "DNF", "why": f"no answer {cap_seconds + 60:.0f} s after the start (cap {cap_seconds:.0f} s)"}
    if pr.is_alive():
        pr.kill()
        pr.join()
    elif not q.empty():
        out = q.get()
        if out.get("status") in ("TIME_LIMIT", "ITERATION_LIMIT"):
            out["status"] = "DNF (" + out["status"] + ")"
    out["wall_seconds"] = time.perf_counter() - t0
    out["cap_seconds"] = cap_seconds
    out["cores"] = 1
    out["what"] = "reference dual simplex (cpp/src/dual_simplex compiled unchanged, oracle/_ref), the LP of this bench line"
    return out


def cusparse_comparator(lp, timeout_s=240):
    """The "kernel to beat" (BASELINE.md §4): the reference's PDHG attempt re-assembled from cusparseSpMV(CSR_ALG2) on A and
    A^T, element-wise kernels, cublasDdot and a CUDA graph per attempt (scripts/cusparse_pdhg.cu), on a uniformly random
    matrix of this LP's shape, timed on this GPU in a child process.  None when the binary is absent or the LP is not one
    of the square sparse workloads."""
    exe = os.path.join(ROOT, "scripts", "_bin", "cusparse_pdhg")
    if not os.path.exists(exe) or lp.m != lp.n or lp.nnz != 8 * lp.m:
        return None
    try:
        r = subprocess.run([exe, str(lp.m)], capture_output=True, text=True, timeout=timeout_s)
        for line in r.stdout.splitlines():
            if line.startswith("{"):
                return json.loads(line)
    except Exception as e:  # noqa: BLE001
        return {"comparator": "cusparse_pdhg", "error": str(e)[:200]}
    return None


DUMP_SAMPLE = 1 << 21  # entries kept of a longer solution vector: 2 x 16 MB at float64


def dump_outputs(out_dir, st, x, y):
    """Writes one step's results as <out_dir>/<name>.npy so that two builds can be compared output for output.  A
    vector longer than DUMP_SAMPLE is cut to the entries at the same seeded random positions on every run."""
    os.makedirs(out_dir, exist_ok=True)

    def sample(v):
        v = np.asarray(v, np.float64)
        if v.size <= DUMP_SAMPLE:
            return v
        return v[np.sort(np.random.default_rng(0).choice(v.size, DUMP_SAMPLE, replace=False))]

    arrays = {"primal_solution": sample(x), "dual_solution": sample(y)}
    for name in ("primal_objective", "dual_objective", "relative_gap", "l2_relative_primal_residual",
                 "l2_relative_dual_residual", "number_of_steps_taken"):
        arrays[name] = np.array([getattr(st, name)], np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_reference(args):
    """CPU arm: the reference's PDLP as restated by the oracle port, all host threads, bounded sample."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = usable_cores()
    os.environ["OMP_NUM_THREADS"] = str(cores)  # torchrun presets 1; must be set before the OpenMP runtime starts
    lp = workload(args)
    sample = args.cpu_iters
    for _ in range(max(0, args.warmup - 1)):
        pass  # the warm-up of this arm is the untimed initialisation + 12 iterations of time_cpu_oracle
    v, per = time_cpu_oracle(lp, cores, sample, args.steps)
    dt = per * args.steps
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config_dict(args, lp, 1),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{sample} PDLP iterations per step of the same LP (oracle/pdlp_oracle.cpp, OpenMP)"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--workload", default="c4", choices=["c4", "c2", "c3"])
    ap.add_argument("--rows", type=int, default=0, help="override the workload's row count (sparse_lp workloads)")
    ap.add_argument("--cols", type=int, default=0)
    ap.add_argument("--nnz-per-row", type=int, default=8)
    ap.add_argument("--locality", type=float, default=0.0, help="column-locality knob rho of the sparse workloads")
    ap.add_argument("--iters", type=int, default=ITERS_PER_STEP)
    ap.add_argument("--cpu-iters", type=int, default=0,
                    help="oracle iterations per step (CPU arm / cpu_baseline); 0 = sized to ~20 s from the nnz count")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--gap-iteration-limit", type=int, default=400000,
                    help="iteration cap of the untimed time-to-1e-6-gap solve reported in detail (0 = skip)")
    ap.add_argument("--gap-time-limit", type=float, default=150.0, help="time cap (s) of that solve")
    ap.add_argument("--profile-reps", type=int, default=200)
    ap.add_argument("--simplex-cap", type=float, default=20.0,
                    help="seconds given to the reference's own CPU path (dual simplex, 1 core) on this LP; 0 = skip")
    ap.add_argument("--comparator", default="auto", choices=["auto", "off"],
                    help="time the cuSPARSE/cuBLAS re-assembly of the reference's attempt (scripts/cusparse_pdhg.cu) beside ours")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned to its caller as DIR/<name>.npy (float64): primal and "
                         "dual solution (a fixed, seeded sample of DUMP_SAMPLE entries when longer), objectives, residuals "
                         "and the iteration count; rank 0 only, so at N > 1 the dual is rank 0's block of rows")
    args = ap.parse_args()
    if args.cpu_iters <= 0:  # the OpenMP oracle runs roughly 1e8 nonzeros/s of PDHG iteration on 8 cores
        nnz_guess = {"c4": 80e6, "c2": 8e6, "c3": 0.9e6}[args.workload]
        args.cpu_iters = int(max(4, min(400, 1.5e8 / nnz_guess * 4)))
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup

    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from cuopt_b200 import capi

    lp = workload(args)
    settings = capi.Settings(method=capi.CUOPT_METHOD_PDLP, log_to_console=False, iteration_limit=args.iters)
    settings.set("optimality_tolerance", 0.0)  # never stop early: every step runs exactly `iters` iterations

    comm = None
    shard = None
    if world > 1:
        from cuopt_b200 import dist as cdist
        comm = cdist.bootstrap(rank, world, device=torch.device("cuda", local))
        shard = cdist.shard_rows(lp, rank, world)
        shard = shard[:2] + tuple(np.ascontiguousarray(a) for a in shard[2:])

    gsol_status = [None]

    def one_step():
        # e2e path: HOST numpy buffers -> C ABI -> HOST result buffers
        if world == 1:
            p = capi.Problem.create_ranged(lp.offsets, lp.indices, lp.values, lp.con_lb, lp.con_ub, lp.c, lp.var_lb,
                                           lp.var_ub)
            sol = capi.solve(p, settings)
        else:  # this rank's block of constraint rows (host arrays cut once, outside the timed region); collective solve
            _, _, off, idx, val, clb, cub = shard
            p = capi.Problem.create_ranged(off, idx, val, clb, cub, lp.c, lp.var_lb, lp.var_ub)
            sol = capi.solve_distributed(p, settings, comm)
        if sol.return_code != 0:
            raise RuntimeError(sol.error_string)
        x = sol.primal(); y = sol.dual()
        st = sol.stats()
        gsol_status[0] = sol.termination_reason
        return st, (x, y)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        one_step()
    sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sampler.start()
    t0 = time.perf_counter()
    its = 0; dev_s = 0.0; launches = 0; setup_s = 0.0; loop_s = 0.0; term_s = 0.0
    for _ in range(args.steps):
        st, last_xy = one_step()
        its += st.number_of_steps_taken
        dev_s += st.pdhg_loop_seconds + st.termination_seconds
        loop_s += st.pdhg_loop_seconds; term_s += st.termination_seconds
        setup_s += st.setup_seconds
        launches += st.kernel_launches
    barrier()
    wall = time.perf_counter() - t0
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs and args.steps > 0:
        dump_outputs(args.dump_outputs, st, *last_xy)

    # max over ranks (device time and wall), sum of iterations
    if world > 1:
        t = torch.tensor([dev_s, wall], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_s, wall = float(t[0]), float(t[1])
        c = torch.tensor([launches], dtype=torch.float64, device="cuda")
        dist.all_reduce(c, op=dist.ReduceOp.SUM)
        launches = int(c[0])  # `its` is NOT summed: all ranks iterate on ONE joint LP

    # second half of BASELINE.json's metric: time to a 1e-6 relative gap (all six tolerances 1e-6), one solve through
    # the same call as the timed steps, outside the timed region; collective at N > 1
    to_gap = None
    if args.gap_iteration_limit > 0:
        gs = capi.Settings(method=capi.CUOPT_METHOD_PDLP, log_to_console=False, iteration_limit=args.gap_iteration_limit,
                           time_limit=args.gap_time_limit)
        gs.set("optimality_tolerance", 1e-6)
        saved, settings = settings, gs
        barrier()
        tg = time.perf_counter()
        gst, _ = one_step()
        barrier()
        tg = time.perf_counter() - tg
        settings = saved
        to_gap = {"tolerance": 1e-6, "wall_seconds": tg, "solver_loop_seconds": gst.pdhg_loop_seconds + gst.termination_seconds,
                  "iterations": gst.number_of_steps_taken, "relative_gap": gst.relative_gap,
                  "primal_objective": gst.primal_objective, "planted_optimum": lp.optimal_objective,
                  "dual_objective": gst.dual_objective,
                  "relative_primal_residual": gst.l2_relative_primal_residual,
                  "relative_dual_residual": gst.l2_relative_dual_residual, "status": gsol_status[0],
                  "reached": bool(gsol_status[0] == "Optimal")}

    # roofline of the dominant kernel, measured in situ with CUDA events on the solver's stream
    roof = None
    cpu = None
    extra = {}
    if rank == 0:
        peaks, peak_kind = measured_peaks()
        p = capi.Problem.create_ranged(lp.offsets, lp.indices, lp.values, lp.con_lb, lp.con_ub, lp.c, lp.var_lb, lp.var_ub)
        prof = capi.Solver(p, settings).profile_kernels(120, args.profile_reps)
        ks = {"k_primal_step": (prof.ms_primal_step, prof.bytes_primal_step),
              "k_dual_step": (prof.ms_dual_step, prof.bytes_dual_step),
              "k_transpose_step": (prof.ms_transpose_step, prof.bytes_transpose_step)}
        dom = max(ks, key=lambda k: ks[k][0])
        ms, by = ks[dom]
        achieved = by / (ms * 1e-3) / 1e9
        blocks = {"k_dual_step": prof.blocks_dual, "k_transpose_step": prof.blocks_transpose}.get(dom, 1)
        launched_as = dom if blocks <= 1 else (
            f"{blocks - 1} x k_block_pass + {dom}<INIT> on the last column block (gather blocking: the step's product is split "
            "by column blocks, the row epilogue is fused into the last block's pass; timed as one group)")
        # DRAM traffic of that step from the committed `ncu --set full` capture of the same workload (bytes per step)
        traffic, traffic_src = NCU_TRAFFIC.get((args.workload, dom, blocks > 1), (None, None))
        roof = {"bound": "hbm", "kernel": dom, "launched_as": launched_as, "achieved": achieved, "peak": peaks["hbm_gbs"],
                "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"], "traffic": traffic,
                "traffic_source": None if traffic is None else f"committed capture: {traffic_src}",
                "peak_source": peak_kind, "algorithmic_bytes_per_launch": by, "ms_per_launch": ms,
                "measured_on": "1 GPU, the full LP" + ("" if world == 1 else
                               f" (a probe on rank 0's GPU beside the {world}-GPU run: the sharded attempt runs other kernels on 1/{world} of the rows; see detail.kernels)")}
        # second bound of the SpMV steps (profiles/r2/request_port_roofline.md): every gathered double of a random column is one
        # L1TEX miss request and an SM sends at most one request per clock towards L2
        try:
            sm_count = torch.cuda.get_device_properties(local).multi_processor_count
            sm_hz = 1e6 * float((clocks or {}).get("sm_mhz") or (clocks or {}).get("sm_max_mhz") or 1965.0)
            floor_ms = 1e3 * (lp.nnz + (12 * lp.nnz) / 128.0) / (sm_count * sm_hz)  # gathers + coalesced 128-byte stream requests
            roof["request_port"] = {"what": "L1TEX -> crossbar requests: 1 per clock per SM; one per gathered double + one per 128 B of matrix stream",
                                    "floor_ms_per_launch": floor_ms, "frac_of_floor": floor_ms / ms if dom != "k_primal_step" else None}
        except Exception:  # noqa: BLE001
            pass
        b_iter = lp.algorithmic_bytes_per_iteration()
        extra = {"kernels": {k: {"ms": v[0], "algorithmic_GBps": v[1] / (v[0] * 1e-3) / 1e9} for k, v in ks.items()},
                 "iteration": {"ms_in_batch": prof.ms_iteration, "algorithmic_bytes": b_iter,
                               "algorithmic_GBps": b_iter / (prof.ms_iteration * 1e-3) / 1e9,
                               "frac_of_hbm_peak": b_iter / (prof.ms_iteration * 1e-3) / 1e9 / peaks["hbm_gbs"]},
                 "grids": {"primal": prof.grid_primal, "dual": prof.grid_dual, "transpose": prof.grid_transpose},
                 "setup_seconds_per_step": setup_s / args.steps, "time_to_gap": to_gap}
        if args.comparator == "auto" and world == 1:
            comp = cusparse_comparator(lp)
            if comp is not None:
                if "us_attempt_graph" in comp:
                    comp["ours_us_attempt_in_batch"] = 1e3 * prof.ms_iteration
                    comp["ours_vs_comparator"] = comp["us_attempt_graph"] / (1e3 * prof.ms_iteration)
                extra["cusparse_comparator"] = comp
    if rank == 0 and args.workload == "c3":
        # the reference's own CPU path on this LP (dual simplex, 1 core), from the committed fixture — not re-timed here
        try:
            with open(os.path.join(ROOT, "tests", "golden", "c3_reference_simplex.json")) as f:
                extra["reference_dual_simplex"] = [c for c in json.load(f)["cases"] if c["rows"] == lp.m][0]
        except Exception:  # noqa: BLE001
            pass
    if rank == 0:
        extra["solver_seconds_per_step"] = {"pdhg_batches": loop_s / args.steps, "major_iterations": term_s / args.steps}
        extra["transport"] = os.environ.get("CUOPT_B200_DIST_MODE", "gather") if world > 1 else None
        if not args.no_cpu_baseline and world == 1:  # the CPU baseline is timed at N = 1 only
            cores = usable_cores()
            os.environ["OMP_NUM_THREADS"] = str(cores)
            v_cpu, _ = time_cpu_oracle(lp, cores, args.cpu_iters, 3)
            cpu = {"value": v_cpu, "unit": UNIT, "cores": cores, "kind": "port",
                   "sample": f"3 x {args.cpu_iters} PDLP iterations of the same LP by oracle/pdlp_oracle.cpp (OpenMP), after "
                             "12 untimed iterations (same protocol as --impl reference)"}
        if args.simplex_cap > 0 and world == 1:
            extra["reference_cpu_path"] = reference_dual_simplex_leg(lp, args.simplex_cap)

    if rank == 0:
        h2d = 12 * lp.nnz + 4 * (lp.m + 1) + 8 * (3 * lp.n + 2 * lp.m)  # A once (A^T is built on the device) + c,l,u,lc,uc
        d2h = 8 * (2 * lp.n + lp.m)
        out = {"metric": METRIC, "value": its / dev_s, "unit": UNIT, "n_gpus": world, "steps": args.steps,
               "warmup": args.warmup, "ms_per_step": 1e3 * wall / args.steps, "higher_is_better": True,
               "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
               "config": config_dict(args, lp, world), "clocks": clocks,
               "e2e": {"value": its / wall, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
               "gpu_launches": launches, "roofline": roof, "cpu_baseline": cpu, "detail": extra}
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
