#!/usr/bin/env python
"""bench.py — headline benchmark of the SVSDF cost+gradient hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A *step* is one pass of the hot path over one batch of synthetic input: one evaluation of
TrajOptimizer::addSaftyPenaOnSweptVolumeParallelTrueSDF (reference: back_end_optimizer.hpp:774-869) over the
200 000 query points of BASELINE config 2 (star shape, 8-piece MINCO), i.e. what the outer optimiser calls once
per cost evaluation.  For N > 1 (launched by torchrun, one rank per GPU) every rank evaluates its own problem of
the same size (batch-of-problems mode, weak scaling); the shared map is broadcast once over NCCL before timing and
there is no collective on the data path.

Reported on ONE JSON line by rank 0:
  value            whole-job query points / second, inputs resident in HBM, device time (CUDA events on the
                   launching stream, max over ranks)
  e2e              the same metric through the C ABI with HOST buffers (svsdf_set_points + svsdf_cost_grad:
                   host->device copy of the points and of the trajectory, device->host copy of cost/gradients inside
                   the timed region)
  lbfgs            full L-BFGS optimisation from x0 through svsdf_optimize (iterations/s, evaluations/s)
  roofline         FP64 (non-tensor) roofline of the dominant kernel k_outer: achieved = flop_per_launch / t, with
                   flop_per_launch (DADD + DMUL + 2 DFMA thread instructions) from the committed ncu capture of the same
                   workload (profiles/r2_k_outer_roofline.json, scripts/roofline_from_ncu.py) and t measured here with
                   CUDA events; the capture's FP64-pipe-active and issue-active percentages are reported next to it
  cpu_baseline     the reference's CPU path timed on this box's host cores: the reference's OWN code compiled where it
                   lies (oracle/_ref/libref_path_glibc.so, kind "reference") when that library travelled with the
                   snapshot, else the line-for-line restatement under oracle/ (kind "port")
`--impl reference` times that CPU path alone on the same workload with the same metric / config keys.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

P_POINTS = 200_000
N_PIECES = 8
SHAPE = "star"
ROOFLINE_JSON = os.path.join(ROOT, "profiles", "r2_k_outer_roofline.json")  # ncu-derived, scripts/roofline_from_ncu.py
METRIC = "svsdf_query_pts_per_sec"
UNIT = "pts/s"


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append((time.time(), ln.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [ln for (ts, ln) in self.lines if t0 - 0.05 <= ts <= t1 + 0.15] or [ln for (_, ln) in self.lines]
        sm, mx, reasons = [], [], set()
        for ln in rows:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def build_problem(rank: int):
    """Config 2 for every rank: each process builds the scene BASELINE.json states into its own host and device buffers — an
    independent replica whose work equals config 2's exactly, so that the per-GPU work is fixed as N grows (weak scaling) and the
    max over ranks measures the box.  (A cyclic shift of the point order was tried to make the replicas differ: it moves the batch
    boundaries and costs the shifted ranks 3.5 % — a different workload, not a slower GPU.  Batches of genuinely different problems
    are measured by scripts/run_batch.py, BASELINE config 5.)"""
    from implicit_svsdf_planner_b200 import scenes

    return scenes.make_scene(SHAPE, N_PIECES, P_POINTS)


def workload_config(world: int) -> dict:
    """The `config` object of the JSON line: identical for both arms (the driver compares them)."""
    return {
        "workload": "config2: star, 8-piece MINCO, 200k query points, one cost+gradient evaluation per step"
                    + ("" if world == 1 else f"; {world} independent replicas of it in flight, one per GPU (own process, own host and device buffers)"),
        "shape": SHAPE, "pieces": N_PIECES, "points_per_gpu": P_POINTS, "problems": world,
        "l2": "GPU arm: flushed between timed iterations (320 MB memset, untimed), inputs are 3.2 MB; CPU arm: n/a",
        "parallelism": "one problem per GPU, no data-path collective" if world > 1 else "single GPU",
    }


def thread_candidates(nproc: int):
    c = {int(round(1.5 * nproc)), nproc, max(1, nproc // 2), max(1, nproc // 4)}
    return sorted(c, reverse=True)


class CpuPath:
    """The reference's CPU implementation of the path, two builds of the same algorithm (results bit-identical per point,
    tests/test_oracle_ref_pin.py): "reference" = its own code compiled where it lies (oracle/_ref; the Eigen it is compiled
    against is the stand-in of oracle/ref_shim, since Eigen itself is not in this image) and "port" = the plain-C++ restatement under
    oracle/ (no Eigen temporaries — about 2-4x faster per point).  Both run the OpenMP loop with schedule(dynamic); the FASTER
    of the two is reported as the CPU figure (never understate the CPU), the other beside it."""

    WHAT = {"reference": "the reference's own source (Shape.hpp classes, trajectory.hpp, minco.hpp, the SweptVolumeManager queries and the "
                         "addSaftyPenaOnSweptVolumeParallelTrueSDF OpenMP loop, cut verbatim / included whole) compiled -O3 against the Eigen "
                         "stand-in of oracle/ref_shim into oracle/_ref/libref_path_glibc.so",
            "port": "line-for-line plain-C++ restatement under oracle/ (glibc sin/cos, -O3 -fopenmp), bit-identical per point to the reference build"}

    def __init__(self, sc, kind=None):
        from oracle import oracle_py as O
        from oracle import ref_py as R

        self.nproc = O.num_procs()
        self.sc = sc
        self.co = sc.coeffs_colmajor()
        if kind is None:
            kind = "reference" if R.available("glibc") else "port"
        self.kind = kind
        self.what = self.WHAT[kind]
        if kind == "reference":
            self.h = R.RefPath(sc.shape, weight_p=sc.weight_p, safety_hor=sc.safety_hor, rho=sc.rho, threads=1, variant="glibc")
        else:
            self.h = O.Oracle(sc.shape, weight_p=sc.weight_p, safety_hor=sc.safety_hor, rho=sc.rho, threads=1, variant="glibc")
        self.h.set_points(sc.points)

    @staticmethod
    def kinds():
        from oracle import ref_py as R

        return ["reference", "port"] if R.available("glibc") else ["port"]

    @staticmethod
    def fastest(sc, reps: int = 3):
        """(CpuPath with its best thread count set, seconds per evaluation, record of everything tried)"""
        best, tried_all = None, {}
        for kind in CpuPath.kinds():
            cp = CpuPath(sc, kind)
            th, tried = cp.pick_threads(reps)
            tried_all[kind] = {"threads": th, "seconds_per_eval": tried[th], "pts_per_s": sc.P / tried[th],
                               "tried_s_per_eval": {str(k): round(v, 4) for k, v in tried.items()}}
            if best is None or tried[th] < best[1]:
                best = (cp, tried[th], th)
        return best[0], best[1], best[2], tried_all

    def eval_once(self):
        return self.h.cost_grad(self.sc.T, self.co)

    def pick_threads(self, reps: int = 3):
        """README tip: threads = 1.5 x logical cores; that oversubscribes many-core hosts, so a few counts are tried
        (best of `reps` each) and the fastest is used."""
        tried = {}
        for th in thread_candidates(self.nproc):
            self.h.set_threads(th)
            self.eval_once()
            best = float("inf")
            for _ in range(reps):
                t0 = time.perf_counter()
                self.eval_once()
                best = min(best, time.perf_counter() - t0)
            tried[th] = best
        th = min(tried, key=tried.get)
        self.h.set_threads(th)
        return th, tried

    def lbfgs(self, max_iterations: int):
        """The product's host L-BFGS (same solver, same parameters as the GPU arm) minimising the CPU path's own cost callback
        (costFunctionLmbmParallel of the reference when kind == "reference")."""
        from implicit_svsdf_planner_b200 import api

        sc = self.sc
        self.h.set_conditions(sc.init_s, sc.final_s, sc.N)
        n_eval = [0]

        def fun(x):
            n_eval[0] += 1
            return self.h.evaluate(x)

        params = api.default_lbfgs_params(mem_size=16, past=3, delta=1e-6, g_epsilon=0.0, max_iterations=max_iterations, min_step=1e-32)
        t0 = time.perf_counter()
        res = api.lbfgs_minimize(fun, sc.x0, params)
        dt = time.perf_counter() - t0
        rc, x, st = res[0], res[1], res[2]
        return {"iters_per_sec": st["iterations"] / dt, "evals_per_sec": n_eval[0] / dt, "iterations": st["iterations"],
                "evaluations": n_eval[0], "status": rc, "final_cost": st["final_cost"], "seconds": dt, "max_iterations": max_iterations}


def cpu_baseline(sc, reps: int = 3):
    """cpu_baseline leg of the GPU arm's line (rank 0, N = 1): the CPU path on the FULL config-2 workload."""
    cp, sec, th, tried = CpuPath.fastest(sc, reps)
    return {"value": sc.P / sec, "unit": UNIT, "cores": cp.nproc, "threads": th, "kind": cp.kind, "what": cp.what,
            "sample": f"the whole {sc.P}-point config-2 workload, one cost+gradient evaluation, best of {reps} after 1 warm-up, OpenMP "
                      "schedule(dynamic), best of the thread counts {1.5, 1, 1/2, 1/4} x nproc; the faster of the two builds of the CPU path "
                      "is reported, both are in `builds`",
            "builds": tried, "seconds_per_eval": sec}


def dump_outputs(outdir: str, cost, grad_T, grad_coeffs, n_inside=None):
    """The arrays a caller of the timed path receives, one float64 .npy each (a few hundred bytes for config 2)."""
    os.makedirs(outdir, exist_ok=True)
    arrays = {"cost": np.atleast_1d(cost), "grad_T": grad_T, "grad_coeffs": grad_coeffs}
    if n_inside is not None:
        arrays["n_inside"] = np.atleast_1d(n_inside)
    for name, a in arrays.items():
        np.save(os.path.join(outdir, name + ".npy"), np.asarray(a, dtype=np.float64).reshape(-1))


def run_reference(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return 0
    sc = build_problem(0)
    cp, _, threads, tried = CpuPath.fastest(sc, 3)  # the faster of the two builds of the reference's CPU path, best thread count
    for _ in range(args.warmup):
        cp.eval_once()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res = cp.eval_once()
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, res[0], res[1], res[2])
    value = sc.P * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cp.nproc, "threads": threads, "kind": cp.kind, "what": cp.what,
                         "sample": f"each step = one cost+gradient evaluation of the whole {sc.P}-point config-2 workload (rank 0 only; at N > 1 the "
                                   "GPU arm runs N such problems concurrently, this arm runs one); the faster of the two builds of the CPU path at its "
                                   "best thread count (best of 3 per count), see `builds`",
                         "builds": tried},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if not args.no_lbfgs:
        line["lbfgs"] = cp.lbfgs(max_iterations=4)  # bounded: a handful of iterations, ~20 evaluations of 200k points
    print(json.dumps(line), flush=True)
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-lbfgs", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (cost, gradients, inside count) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    from implicit_svsdf_planner_b200 import api, batch

    rank, world, local = dist_env()
    torch.cuda.set_device(local)
    numa_cpus = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        numa_cpus = batch.bind_to_gpu_numa(local)  # before any pinned buffer exists (the e2e leg's staging memory)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    # Every rank runs its OWN replica of config 2 (own process, own host and device buffers, equal work): per-GPU work and per-rank
    # working set are the same at every N (weak scaling), so the max over ranks measures the box.  At N = 1 this is config 2 alone.
    sc = build_problem(rank)
    co = sc.coeffs_colmajor()
    # the only shared datum of the batch mode is the map: broadcast it once from rank 0 (NCCL) before timing
    map_bytes = None
    if world > 1:
        kern = batch.pack_map_kernel_from_points(sc.points, sc.resolution) if rank == 0 else None
        map_bytes = int(batch.broadcast_map(kern, device=torch.device("cuda", local)).numel())

    strict = os.environ.get("SVSDF_BENCH_FMA", "0") != "1"  # default: the bit-exact strict build
    ctx = api.Context(SHAPE, weight_p=sc.weight_p, safety_hor=sc.safety_hor, rho=sc.rho, device=local, strict_fp=strict)
    ctx.set_points(sc.points)
    ctxs = [ctx]

    def problem_of(step):
        return sc, ctx, co
    flush = torch.empty(160 * 1024 * 1024, dtype=torch.float16, device=f"cuda:{local}")  # 320 MB > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    # ---- device-resident throughput (value) ----
    for w in range(args.warmup):
        pr, c, cc = problem_of(w)
        c.cost_grad_device(pr.T, cc, repeats=1, fetch=False)
    launches0 = sum(c.kernel_launches() for c in ctxs)
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)
    barrier()
    t_wall0 = time.time()
    ms_steps, outer_ms = [], []
    for s_ in range(args.steps):
        pr, c, cc = problem_of(s_)
        flush.zero_()  # flush L2 between timed iterations (untimed)
        torch.cuda.synchronize()
        # every step copies its result to the host after the stop event; fetch only hands the last one to Python
        fetch = bool(args.dump_outputs) and s_ == args.steps - 1
        ms, out = c.cost_grad_device(pr.T, cc, repeats=1, fetch=fetch)  # CUDA events on the launching stream
        ms_steps.append(ms)
        if c is ctx:
            outer_ms.append(c.last_kernel_ms()[1])
    barrier()
    t_wall1 = time.time()
    clocks = sampler.stop(t_wall0, t_wall1)
    launches = sum(c.kernel_launches() for c in ctxs) - launches0
    my_ms = float(sum(ms_steps))
    t = torch.tensor([my_ms], dtype=torch.float64, device=f"cuda:{local}")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    value = world * sc.P * args.steps / (total_ms * 1e-3)
    # per-rank view (diagnostic: the max over ranks above is set by the slowest GPU of the box)
    per_rank = torch.zeros(world, 2, dtype=torch.float64, device=f"cuda:{local}")
    per_rank[rank, 0] = my_ms / args.steps
    per_rank[rank, 1] = float(clocks.get("sm_mhz") or 0.0)
    if world > 1:
        dist.all_reduce(per_rank, op=dist.ReduceOp.SUM)
    per_rank = per_rank.cpu().numpy()

    # ---- end-to-end through the C ABI with host buffers ----
    for w in range(2):
        pr, c, cc = problem_of(w)
        c.set_points(pr.points)
        c.cost_grad(pr.T, cc)
    barrier()
    e0 = time.perf_counter()
    for s_ in range(args.steps):
        pr, c, cc = problem_of(s_)
        c.set_points(pr.points)  # host -> device copy of this step's query points
        cost, gT, gC = c.cost_grad(pr.T, cc)  # host trajectory in, host cost/gradients out
    torch.cuda.synchronize()
    e_ms = 1e3 * (time.perf_counter() - e0)
    te = torch.tensor([e_ms], dtype=torch.float64, device=f"cuda:{local}")
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * sc.P * args.steps / (float(te.item()) * 1e-3)
    blob_bytes = 8 * (4 + N_PIECES + 18 * N_PIECES + int(sc.T.sum() / 0.15 + 2))
    h2d = sc.P * 16 + blob_bytes
    d2h = 8 * (1 + 19 * N_PIECES + 1)

    extra = {}
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, out[0], out[1 + 18 * N_PIECES:1 + 19 * N_PIECES], out[1:1 + 18 * N_PIECES], out[1 + 19 * N_PIECES])
    if rank == 0:
        # ---- roofline of the dominant kernel (k_outer), FP64 non-tensor pipe ----
        ctx.executed_evals(True)
        ctx.cost_grad_device(sc.T, co, repeats=1, fetch=False)
        lane_evals = ctx.executed_evals(False)
        peak = ctx.fp64_peak_tflops()
        t_outer = statistics.mean(outer_ms) * 1e-3
        cap = json.load(open(ROOFLINE_JSON)) if os.path.exists(ROOFLINE_JSON) else None
        peaks = {}
        ppath = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(ppath):
            peaks = json.load(open(ppath))
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        alg_bytes = sc.P * 16
        achieved = (cap["flop_per_launch"] / t_outer / 1e12) if cap else None
        extra["roofline"] = {
            "bound": "fp64", "kernel": "k_outer", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
            "frac": (achieved / peak) if achieved else None,
            "peak_source": "DFMA micro-benchmark in this run (svsdf_fp64_peak); MEASURED_PEAKS.json has no FP64 figure",
            "flop_per_launch": cap["flop_per_launch"] if cap else None,
            "flop_source": "profiles/r2_k_outer_roofline.json: DADD + DMUL + 2 DFMA thread instructions of one launch (ncu --set full capture of this workload); "
                           "the strict build issues DMUL + DADD where an FMA build would issue one DFMA, so the DFMA-based peak is reachable "
                           "only at half rate by this instruction mix - see fp64_pipe_active_pct",
            "fp64_pipe_active_pct": cap.get("fp64_pipe_active_pct") if cap else None,
            "issue_active_pct": cap.get("issue_active_pct") if cap else None,
            "traffic": cap.get("dram_bytes_per_launch") if cap else None,
            "evals_per_point_executed": lane_evals / sc.P, "kernel_ms": t_outer * 1e3,
            "flop_per_lane_eval": (cap["flop_per_launch"] / lane_evals) if cap else None,
            "kernel_share_of_step": t_outer * 1e3 / statistics.mean(ms_steps),
            "hbm": {"achieved": alg_bytes / t_outer / 1e9, "peak": hbm_peak, "unit": "GB/s", "frac": alg_bytes / t_outer / 1e9 / hbm_peak,
                    "peak_source": "MEASURED_PEAKS.json (measured)" if peaks else "fallback", "algorithmic_bytes": alg_bytes},
        }
        km = ctx.last_kernel_ms()
        extra["kernel_ms"] = {"k_pose_table": km[0], "k_outer": km[1], "k_compact+k_gsip": km[2], "k_finalize": km[3]}
        # ---- full optimisation to convergence (LBFGS iters/sec part of the metric) ----
        if not args.no_lbfgs:
            params = api.default_lbfgs_params(mem_size=16, past=3, delta=1e-6, g_epsilon=0.0, max_iterations=200, min_step=1e-32)
            rc, x, T, b, st = ctx.optimize(sc.init_s, sc.final_s, sc.x0, sc.N, params)
            # the same small budget the CPU arm runs (`--impl reference`: max_iterations = 4) for a like-for-like evaluations/s ratio
            p4 = api.default_lbfgs_params(mem_size=16, past=3, delta=1e-6, g_epsilon=0.0, max_iterations=4, min_step=1e-32)
            rc4, _, _, _, st4 = ctx.optimize(sc.init_s, sc.final_s, sc.x0, sc.N, p4)
            extra["lbfgs_same_budget_as_cpu_arm"] = {"iters_per_sec": st4["iterations"] / st4["seconds"], "evals_per_sec": st4["evaluations"] / st4["seconds"],
                                                     "iterations": st4["iterations"], "evaluations": st4["evaluations"], "status": st4["status"],
                                                     "final_cost": st4["final_cost"], "seconds": st4["seconds"], "max_iterations": 4}
            extra["lbfgs"] = {"iters_per_sec": st["iterations"] / st["seconds"], "evals_per_sec": st["evaluations"] / st["seconds"],
                              "iterations": st["iterations"], "evaluations": st["evaluations"], "status": st["status"],
                              "final_cost": st["final_cost"], "seconds": st["seconds"], "gpu_seconds": st["gpu_seconds"]}
        if not args.no_cpu_baseline and world == 1:  # rank 0 at N = 1 only
            extra["cpu_baseline"] = cpu_baseline(sc)

    if world > 1:
        dist.barrier()
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "per_rank": {"ms_per_step": [float(v) for v in per_rank[:, 0]], "sm_mhz": [float(v) for v in per_rank[:, 1]]},
            "dtype": "f64", "data": "synthetic",
            "config": workload_config(world),
            "impl_config": {"rank_cpu_affinity": (f"GPU-local NUMA CPUs ({numa_cpus})" if numa_cpus else "unchanged"), "fp_mode": "strict (-fmad=false)" if strict else "fma-contracted (opt-in, not bit-exact)", "map_broadcast_bytes": map_bytes},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": float(te.item()) / args.steps},
            "gpu_launches": launches, "clocks": clocks, "wall_ms_timed_region": 1e3 * (t_wall1 - t_wall0),
        }
        line.update(extra)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
