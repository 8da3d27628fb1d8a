#!/usr/bin/env python
"""Benchmark of the hot path (BASELINE.json): optimised trajectories/s (M2) and constraint+Jacobian
evaluations/s (M1).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N ...            # the reference's CPU path (scipy SLSQP + its closures)

Prints ONE JSON line (rank 0).  Headline workload: config C4 of BASELINE.json, batched 3-D safe-flight-corridor
trajectories x 262,144 problems per GPU (the configuration the north star quotes its trajectory target on and the
largest single-GPU configuration).  A "step" is one pass of the hot path over one batch: every problem of the batch
is solved from its initial guess.  The same line carries one sub-record per other BASELINE configuration under
`configs` (C1 single-problem latency through the drop-in class; C2 and C3 at their full batch sizes; C5 as a STRONG
sweep: 1,048,576 bicycle/unicycle problems in total, sharded over the ranks by distributed.solve_sharded), each
with its own value, e2e, roofline and -- on one GPU -- parity sample against the CPU reference.

Multi-GPU: one process per GPU (torchrun), independent problems sharded by rank (weak scaling for the headline:
every rank owns a full batch with its own seed), no collective inside the solve, one NCCL all-gather of the result
rows at the end of each step (distributed.all_gather_rows).
"""
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

# dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed
# `ncu --set full` captures (profiles/README.md), per problem the launch worked through
NCU_TRAFFIC_PER_PROBLEM = {}
NCU_TRAFFIC_EVAL_PER_EVAL = {}
NCU_TRAFFIC_SAMPLE_PER_SAMPLE = {}
try:
    with open(os.path.join(ROOT, "profiles", "traffic.json")) as _f:
        _t = json.load(_f)
    NCU_TRAFFIC_PER_PROBLEM = _t.get("qp_kernel_bytes_per_problem", {})
    NCU_TRAFFIC_EVAL_PER_EVAL = _t.get("eval_kernel_bytes_per_evaluation", {})
    NCU_TRAFFIC_SAMPLE_PER_SAMPLE = _t.get("sample_kernel_bytes_per_sample", {})
except Exception:
    pass

METRIC = "optimized_trajectories_per_sec"
UNIT = "trajectories/s"
L2_FLUSH_BYTES = 512 << 20
HEADLINE = "C4"
C5_TOTAL = 1048576

WORKLOAD = {"C2": "batched 2D obstacle avoidance (test_obstacle_trajectory_2D shape, 8 circular obstacles) x %d problems per GPU",
            "C3": "batched 2D intermediate-waypoint trajectories with curvature + velocity bounds x %d problems per GPU",
            "C4": "batched 3D safe-flight-corridor trajectories (test_sfc_trajectory_3D shape, 4 corridor boxes) x %d problems per GPU",
            "C5a": "bicycle/unicycle kinematic trajectories, angular-rate + acceleration bounds x %d problems per GPU",
            "C5c": "bicycle/unicycle kinematic trajectories, curvature + acceleration bounds x %d problems per GPU"}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5,
                    help="timed steps of the headline solve and of its evaluation and sampling records; the secondary "
                         "records time fewer so the run stays short: the other configurations and the end-to-end record "
                         "min(steps, 2), the other Jacobian mode 2, C1 5 calls")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default=HEADLINE, help="headline workload: C4 (default) | C2 | C3 | C5a | C5c")
    ap.add_argument("--batch", type=int, default=None, help="problems per GPU (default: the config's full batch)")
    ap.add_argument("--jacobian", default="fd", choices=["analytic", "fd"],
                    help="fd (default): scipy's forward differences emulated on the GPU -- the mode that follows the reference's "
                         "iterates; analytic: closed-form Jacobians (reported next to it as analytic_mode)")
    ap.add_argument("--cpu-sample", type=int, default=None, help="problems in the CPU sample (default: scaled to the host's cores)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="headline only: no sub-records for the other BASELINE configurations")
    ap.add_argument("--fused", action="store_true", help="one persistent solve kernel instead of lock-step stage kernels")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of the headline solve returned (x, f, status, nit, violation of "
                         "rank 0's batch) as DIR/<name>.npy in float64; batches whose outputs exceed 64 MB are "
                         "represented by a fixed, seeded sample of problems")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def config_dict(name, B, L=None, jacobian="fd"):
    """The `config` object: identical in both arms (the reference arm solves a bounded sample of this workload)."""
    from trajectory_generator_b200 import synthetic
    c = {"workload": WORKLOAD[name] % B, "config": name, "problems_per_gpu": int(B), "maxiter": 100, "ftol": 1e-6,
         "objective": synthetic.OBJECTIVE[name], "jacobian": "2-point finite differences (scipy's rule)" if jacobian == "fd" else jacobian,
         "l2": "flushed between iterations (512 MiB fill)",
         "multi_gpu": "independent problems sharded by rank, one NCCL all-gather of result rows per step"}
    return c


def make_batch(name, B, rank=0):
    from trajectory_generator_b200 import synthetic
    gen = {"C2": synthetic.make_c2, "C3": synthetic.make_c3, "C4": synthetic.make_c4}.get(name)
    if gen is not None:
        return gen(B, seed=synthetic.SEED0 + int(name[1]) + 1000 * rank)
    return synthetic.make_c5(B, "angular_rate" if name == "C5a" else "curvature", seed=synthetic.SEED0 + 5 + 1000 * rank)


# --------------------------------------------------------------------------------------------------------------
# CPU path: the reference's scipy SLSQP call on its own closures (oracle/tg_oracle.py restates the Python closures,
# the native steps run in the reference's own C++ compiled unmodified when oracle/_ref exists).  Worker processes
# receive their problems and build the closures BEFORE the clock starts; the product's CUDA library is never
# loaded on this path (synthetic.Batch resolves its layout lazily; containers are plain dataclasses).
# --------------------------------------------------------------------------------------------------------------
def cpu_path_available():
    ref = os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libTrajectoryConstraints.so"))
    port = os.path.exists(os.path.join(ROOT, "oracle", "_build", "libtg_oracle.so"))
    return "ref" if ref else ("oracle" if port else None)


def _cpu_worker_main(conn, name, sub, local_indices, native_kind):
    import warnings
    warnings.simplefilter("ignore")
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import scipy.optimize  # noqa: F401
    import tg_oracle
    from trajectory_generator_b200 import synthetic
    probs = []
    for i in local_indices:
        d, cc, kw = synthetic.container_for(sub, i)
        op = tg_oracle.OracleProblem(d, cc, kw.get("objective_function_type", synthetic.OBJECTIVE[name]),
                                     kw.get("num_intervals_free_space"), native_kind=native_kind)
        probs.append((i, op, op.x0.copy()))
    conn.send("ready")
    while True:
        msg = conn.recv()
        if msg[0] == "stop":
            break
        perturb = msg[1]
        out = []
        for i, op, x0 in probs:
            # perturb = +1 / -1: the same reference solve started one unit in the last place above / below x0 (its own
            # reproducibility)
            op.x0 = np.nextafter(x0, np.inf * perturb) if perturb else x0
            t = time.perf_counter()
            res = op.solve()
            out.append((i, int(res.status), int(res.nit), time.perf_counter() - t, res.x.tolist()))
        conn.send(out)
    conn.close()


class CpuPool:
    """Process pool over the host cores; each worker owns a fixed slice of the sample."""

    def __init__(self, name, sub_batch, procs):
        import multiprocessing as mp
        self.kind = cpu_path_available()
        if self.kind is None:
            raise RuntimeError("oracle libraries are not built (run __graft_entry__.build())")
        n = len(sub_batch)
        chunks = [list(range(n))[k::procs] for k in range(procs)]
        chunks = [c for c in chunks if c]
        ctx = mp.get_context("spawn")
        self.workers = []
        # one process per core, so every process runs its BLAS single-threaded: with the default (one OpenBLAS thread
        # per core in EVERY process) 16 workers x 16 threads fight over 16 cores and the same solves take ~50x longer
        saved = {k: os.environ.get(k) for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS")}
        os.environ.update({k: "1" for k in saved})
        for c in chunks:
            a, b = ctx.Pipe()
            p = ctx.Process(target=_cpu_worker_main, args=(b, name, sub_batch.take(c), list(range(len(c))), self.kind), daemon=True)
            p.start()
            self.workers.append((p, a, c))
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
        for p, a, c in self.workers:
            assert a.recv() == "ready"
        self.cores = len(self.workers)

    def run(self, perturb=0):
        """One pass over the sample.  Returns (seconds, results sorted by problem index)."""
        t = time.perf_counter()
        for p, a, c in self.workers:
            a.send(("go", perturb))
        res = []
        for p, a, c in self.workers:
            part = a.recv()
            res += [(c[r[0]],) + tuple(r[1:]) for r in part]          # worker-local index -> index in the sample
        dt = time.perf_counter() - t
        return dt, sorted(res)

    def close(self):
        for p, a, c in self.workers:
            try:
                a.send(("stop",))
            except Exception:
                pass
        for p, a, c in self.workers:
            p.join(timeout=10)


def default_cpu_sample(name, cores):
    """Bounded sample: about 5-15 s of wall time per pass on the box's cores (one core solves ~13 C4, ~7.5 C2, ~2.4 C3
    or ~3.6 C5 problems per second)."""
    per_core = {"C4": 64, "C3": 32, "C2": 64}.get(name, 32)
    return min(1024, max(64, per_core * cores))


def cpu_kind_label(kind):
    # Python closures are the oracle's restatement; with kind 'ref' the native geometry is the reference's own C++
    return "port"


# --------------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag = index, [], set(), False
        self.max_mhz = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [v.strip() for v in out.strip().split(",")]
                self.samples.append(float(f[0])); self.max_mhz = float(f[1])
                for n, v in zip(names, f[2:]):
                    if v.lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def _claim_stdout():
    """Everything libraries print to fd 1 (e.g. NCCL's version banner on the first collective) goes to stderr;
    the returned file object is the real stdout, used for the ONE JSON line."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    return real


def hist(a):
    return {str(k): int(v) for k, v in zip(*np.unique(np.asarray(a), return_counts=True))}


DUMP_LIMIT_BYTES = 64 * 10 ** 6
DUMP_SEED = 20261020


def dump_outputs(path, outputs):
    """Writes the per-problem output tensors as path/<name>.npy in float64 (the int32 ones convert exactly), so that two
    builds can be compared output for output.  When the rows together exceed DUMP_LIMIT_BYTES, every array keeps the same rows:
    a sorted sample drawn with DUMP_SEED, identical from run to run."""
    host = {k: v.cpu().numpy().astype(np.float64) for k, v in outputs.items()}
    B = len(host["x"])
    row_bytes = sum(8 * (a.size // B) for a in host.values())
    rows = min(B, (DUMP_LIMIT_BYTES - 4096) // row_bytes)        # 4 KiB of room for the .npy headers
    idx = np.arange(B) if rows == B else np.sort(np.random.default_rng(DUMP_SEED).choice(B, rows, replace=False))
    os.makedirs(path, exist_ok=True)
    for k, a in host.items():
        np.save(os.path.join(path, k + ".npy"), np.ascontiguousarray(a[idx]))


# --------------------------------------------------------------------------------------------------------------
# reference arm
# --------------------------------------------------------------------------------------------------------------
def reference_arm(args, out_stream):
    name = args.config
    from trajectory_generator_b200 import synthetic
    B = args.batch or synthetic.FULL_BATCH[name]
    cores = os.cpu_count() or 1
    sample = args.cpu_sample or default_cpu_sample(name, cores)
    bt = make_batch(name, B)                       # the b200 arm's rank-0 batch; its first `sample` problems are solved
    pool = CpuPool(name, bt.take(range(sample)), cores)
    times = []
    res = None
    for it in range(args.warmup + args.steps):
        dt, res = pool.run()
        if it >= args.warmup:
            times.append(dt)
    pool.close()
    sec = float(np.mean(times))
    val = sample / sec
    st = [r[1] for r in res]
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_dict(name, B),
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": pool.cores, "kind": cpu_kind_label(pool.kind),
                             "native": "reference C++ (oracle/_ref)" if pool.kind == "ref" else "plain-C oracle",
                             "sample": "first %d problems of the %s batch per step, scipy SLSQP with 2-point finite differences on the "
                                       "reference's closures, one process per core (%d); closures built before the clock" % (sample, name, pool.cores),
                             "step_seconds": times, "status_histogram": hist(st)},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), file=out_stream, flush=True)


# --------------------------------------------------------------------------------------------------------------
# CUDA arm
# --------------------------------------------------------------------------------------------------------------
class Gpu:
    def __init__(self, args):
        import torch
        import torch.distributed as dist
        from trajectory_generator_b200 import _native
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.lib = _native.lib()
        self.flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=self.dev)
        self.args = args

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, fn, steps, warmup, prepare=None):
        """CUDA events on torch's current stream (the stream the library launches on) around every step; L2 flushed
        between steps.  Returns ms per step, max over ranks of the summed step times."""
        torch = self.torch
        ev = []
        self.barrier()
        for it in range(warmup + steps):
            if prepare:
                prepare()
            self.flush.fill_(it & 1)                      # evict L2 between iterations
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record(); fn(); e.record()
            if it >= warmup:
                ev.append((s, e))
        self.barrier()
        tot = torch.tensor([sum(s.elapsed_time(e) for s, e in ev)], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(tot, op=self.dist.ReduceOp.MAX)
        return tot.item() / steps

    def max_over_ranks(self, v):
        t = self.torch.tensor([float(v)], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.item()


def peaks():
    p = {}
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm = float(p.get("hbm_gbs", 6650.0))
    src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in p else "fallback 6.65 TB/s (B200_PROFILING.md)"
    return hbm, src


def bench_config(G, name, B, steps, warmup, full=True):
    """One BASELINE configuration on every rank's own batch (weak scaling).  Returns (record, arrays for parity)."""
    import ctypes
    torch = G.torch
    from trajectory_generator_b200 import _native, batch as tgb, distributed as tgd, synthetic
    args = G.args
    bt = make_batch(name, B, G.rank)
    L = bt.layout
    dev = G.dev
    par = torch.from_numpy(bt.par).to(dev)
    x0 = torch.from_numpy(bt.x0).to(dev)
    x = torch.empty_like(x0)
    bufs = tgb.SolveBuffers(bt.spec, B, dev)
    hbm_peak, peak_src = peaks()

    def solve_step(mode=args.jacobian):
        out = tgb.solve(bt.spec, par, x, jacobian=mode, buffers=bufs, fused=args.fused)
        if G.world > 1:
            tgd.all_gather_rows(tgd.pack_result_rows(torch, x, out["status"], out["nit"], out["violation"], out["f"]), total=G.world * B)

    launches0 = G.lib.tg_launch_count()
    ms_step = G.timed(solve_step, steps, warmup, prepare=lambda: x.copy_(x0))
    solve_launches = (G.lib.tg_launch_count() - launches0) * steps // (steps + warmup)
    if full and args.dump_outputs and G.rank == 0:
        dump_outputs(args.dump_outputs, {"x": x, "f": bufs.f, "status": bufs.status, "nit": bufs.nit,
                                         "violation": bufs.violation})
    value = G.world * B / (ms_step * 1e-3)
    status = bufs.status.cpu().numpy(); nit = bufs.nit.cpu().numpy()
    x_gpu = x.cpu().numpy()
    arrays = {"x": x_gpu, "status": status, "batch": bt}

    # ---- per-kernel share of a step and the dominant kernel's launch duration: one extra solve with CUDA events
    #      around every stage launch on the launching stream (the C library records them)
    stats = (ctypes.c_double * 6)()
    G.lib.tg_set_stage_timing(1)
    x.copy_(x0); G.flush.fill_(1)
    tgb.solve(bt.spec, par, x, jacobian=args.jacobian, buffers=bufs, fused=args.fused)
    torch.cuda.synchronize()
    G.lib.tg_set_stage_timing(0)
    G.lib.tg_last_solve_stats(stats, 6)
    ms_ls, ms_qp, flops_qp, n_ls, n_qp, rounds = [float(v) for v in stats]
    fp64_peak = ctypes.c_double(0.0)
    _native.check(G.lib.tg_measure_fp64_peak(ctypes.byref(fp64_peak)), "tg_measure_fp64_peak")
    solve_bytes = 8 * (L.P + 2 * L.n + 4) * B
    traffic = NCU_TRAFFIC_PER_PROBLEM.get(name)
    rec = {"metric": METRIC, "value": value, "unit": UNIT, "ms_per_step": ms_step, "steps": steps, "warmup": warmup,
           "scaling": "weak", "config": dict(config_dict(name, B, L, args.jacobian)),
           "shape": {"d": L.d, "N": L.N, "n": L.n, "m": L.m, "meq": L.meq, "parameters_per_problem": L.P},
           "solve_stats": {"mean_nit": float(nit.mean()), "max_nit": int(nit.max()), "status_histogram": hist(status)},
           "gpu_launches": int(solve_launches)}
    if not args.fused and ms_qp > 0:
        # algorithmic work of the QP stage, SURVEY.md 8(d): nit (2 n^3 / 3 + 2 m n^2) per trajectory -- the subproblem
        # term of the reference's SLSQP iteration (factor handling + the m x n least-squares reductions), with the
        # measured mean iteration count.  `executed` is what this solver's own QP stage performs instead (counted by the
        # kernel: active rows only, terminal location rows eliminated) -- the definition `achieved` had in round 1.
        per_traj = float(nit.mean()) * (2.0 * L.n ** 3 / 3.0 + 2.0 * L.m * L.n ** 2)
        ach = per_traj * B / (ms_qp * 1e-3) / 1e12
        ach_exec = flops_qp / (ms_qp * 1e-3) / 1e12
        rec["roofline"] = {
            "kernel": "tg_sqp_qp_kernel", "bound": "fp64", "achieved": ach, "peak": fp64_peak.value, "unit": "TFLOP/s",
            "frac": ach / fp64_peak.value,
            "definition": "SURVEY.md 8(d): mean nit x (2 n^3 / 3 + 2 m n^2) flops per trajectory / time in the QP-stage kernel",
            "algorithmic_flops_per_trajectory_survey": per_traj,
            "executed": {"achieved": ach_exec, "frac": ach_exec / fp64_peak.value, "unit": "TFLOP/s",
                         "flops_per_trajectory": flops_qp / B,
                         "note": "fp64 operations the kernel itself counts for the products, factor updates and scans its "
                                 "dual active-set method performs (the round-1 definition of `achieved`)"},
            "traffic": traffic * B if traffic else None,
            "traffic_note": "dram bytes read + written by one launch of the kernel working through the whole batch (round 10 of a "
                            "solve), from the committed ncu --set full capture scaled per problem (profiles/traffic.json)",
            "launches_per_step": int(n_qp), "avg_launch_ms": ms_qp / max(n_qp, 1.0),
            "share_of_step": ms_qp / (ms_ls + ms_qp), "line_search_and_derivative_kernels_ms": ms_ls, "qp_kernel_ms": ms_qp,
            "algorithmic_flops_per_trajectory": flops_qp / B,
            "peak_source": "measured in this run: DFMA kernel, 8 chains per thread, every SM full "
                           "(MEASURED_PEAKS.json has no fp64 figure; nominal 148 x 64 x 2 x 1.965 GHz = 37.2)",
            "hbm": {"achieved": solve_bytes / (ms_step * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                    "frac": solve_bytes / (ms_step * 1e-3) / 1e9 / hbm_peak, "peak_source": peak_src,
                    "note": "algorithmic HBM bytes per trajectory are 8(P + 2n + 4): not the bound"}}
    else:
        rec["roofline"] = {"kernel": "tg_solve_kernel", "bound": "hbm", "achieved": solve_bytes / (ms_step * 1e-3) / 1e9,
                           "peak": hbm_peak, "unit": "GB/s", "frac": solve_bytes / (ms_step * 1e-3) / 1e9 / hbm_peak,
                           "traffic": None, "peak_source": peak_src}

    # ---- e2e: host buffers through the C-ABI (tg_solve_host), copies inside the timed call
    par_pin = tgb.pinned_empty(bt.par.shape); par_pin[:] = bt.par
    x_pin = tgb.pinned_empty(bt.x0.shape)
    e2e_times = []
    for it in range(1 + min(steps, 2)):
        x_pin[:] = bt.x0
        G.barrier()
        t = time.perf_counter()
        tgb.solve_host(bt.spec, par_pin, x_pin, jacobian=args.jacobian, fused=args.fused)
        G.barrier()
        if it > 0:
            e2e_times.append(time.perf_counter() - t)
    del par_pin, x_pin
    e2e_s = G.max_over_ranks(float(np.mean(e2e_times)))
    rec["e2e"] = {"value": G.world * B / e2e_s, "unit": UNIT, "h2d_bytes_per_step": 8 * B * (L.P + L.n),
                  "d2h_bytes_per_step": 8 * B * (L.n + 1) + 4 * B * 3,
                  "api": "tg_solve_host (C-ABI, page-locked host buffers; copies inside the call)"}
    if not full:
        return rec, arrays

    # ---- the other Jacobian mode on the same batch (2 timed steps), reported next to the timed one
    other = "analytic" if args.jacobian == "fd" else "fd"
    other_ms = G.timed(lambda: solve_step(other), 2, 1, prepare=lambda: x.copy_(x0))
    other_status = bufs.status.cpu().numpy(); other_nit = bufs.nit.cpu().numpy()
    arrays["other_x"] = x.cpu().numpy(); arrays["other_status"] = other_status; arrays["other"] = other
    rec[other + "_mode"] = {"value": G.world * B / (other_ms * 1e-3), "unit": UNIT, "ms_per_step": other_ms, "steps": 2,
                            "mean_nit": float(other_nit.mean()), "status_histogram": hist(other_status)}

    # ---- M1: evaluation kernel on the same batch
    xe_h = synthetic.evaluation_points(bt)
    xe = torch.from_numpy(xe_h).to(dev)
    ev_out = {}
    ms_eval = G.timed(lambda: tgb.evaluate(bt.spec, par, xe, out=ev_out), steps, warmup)
    eval_bytes = 8 * (L.n + L.P + L.m + L.m_nl * L.n + 1 + L.n)
    # e2e: host buffers through tg_eval_host -- page-locked buffers (as the contract asks), reused between calls; the
    # library pipelines the batch in chunks (upload / kernel / download overlap)
    hp = {"par": tgb.pinned_empty(bt.par.shape), "x": tgb.pinned_empty(xe_h.shape)}
    hp["par"][:] = bt.par; hp["x"][:] = xe_h
    hout = {k: tgb.pinned_empty(shp) for k, shp in (("f", (B,)), ("g", (B, L.n)), ("c", (B, L.m)), ("jnl", (B, L.m_nl, L.n)))}
    te = []
    for it in range(4):
        G.barrier()
        t = time.perf_counter()
        tgb.evaluate_host(bt.spec, hp["par"], hp["x"], out=hout)
        if it > 0:
            te.append(time.perf_counter() - t)
    eval_e2e = G.world * B / G.max_over_ranks(float(np.mean(te)))
    assert np.array_equal(hout["f"], ev_out["f"].cpu().numpy())
    del hp, hout
    tr_e = NCU_TRAFFIC_EVAL_PER_EVAL.get(name)
    rec["evals"] = {"metric": "constraint_jacobian_evaluations_per_sec", "value": G.world * B / (ms_eval * 1e-3),
                    "unit": "evaluations/s", "ms_per_step": ms_eval, "bytes_per_eval": eval_bytes,
                    "e2e": {"value": eval_e2e, "unit": "evaluations/s", "h2d_bytes_per_step": 8 * B * (L.P + L.n),
                            "d2h_bytes_per_step": 8 * B * (1 + L.n + L.m + L.m_nl * L.n),
                            "api": "tg_eval_host (C-ABI, page-locked host buffers; copies inside the call, pipelined in chunks)"},
                    "roofline": {"kernel": "tg_eval_kernel", "bound": "hbm",
                                 "achieved": eval_bytes * B / (ms_eval * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                 "frac": eval_bytes * B / (ms_eval * 1e-3) / 1e9 / hbm_peak,
                                 "traffic": tr_e * B if tr_e else None, "peak_source": peak_src}}
    del ev_out

    # ---- f1: output sampling of the solved batch (positions) -- a pure HBM-write stream
    from trajectory_generator_b200 import matrix_evaluation as tgs
    SAMPLES = 1024
    samp = torch.empty((B, L.d, SAMPLES), dtype=torch.float64, device=dev)
    ms_samp = G.timed(lambda: tgs.sample_batch((x, L.d, L.N), num_points=SAMPLES, out=samp), steps, warmup)
    samp_bytes = 8 * L.d * SAMPLES * B + 8 * (L.d * L.N) * B
    tr_s = NCU_TRAFFIC_SAMPLE_PER_SAMPLE.get(str(L.d))
    rec["sampling"] = {"metric": "trajectory_samples_per_sec", "value": G.world * B * SAMPLES / (ms_samp * 1e-3),
                       "unit": "samples/s", "ms_per_step": ms_samp, "samples_per_trajectory": SAMPLES,
                       "roofline": {"kernel": "tg_sample_kernel", "bound": "hbm",
                                    "achieved": samp_bytes / (ms_samp * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                    "frac": samp_bytes / (ms_samp * 1e-3) / 1e9 / hbm_peak,
                                    "traffic": tr_s * B * SAMPLES if tr_s else None,
                                    "bytes_per_sample": 8 * L.d, "peak_source": peak_src}}
    return rec, arrays


def parity_against_cpu(name, arrays, sample, cores, jacobian):
    """CPU baseline on the box's host cores + parity of the CUDA solutions on the same problems (rank 0, N = 1)."""
    bt = arrays["batch"]
    L = bt.layout
    pool = CpuPool(name, bt.take(range(sample)), cores)
    try:
        dt, res = pool.run()
        # how reproducible the reference is against ITSELF: the same scipy solves started from x0 + 1 ulp and from
        # x0 - 1 ulp.  Its forward differences (h = 1.5e-8) amplify last-place differences of the closures by 1/h, so long
        # solves separate; agreement of the CUDA path is therefore also reported on the problems whose reference
        # solution is stable to 1e-5 under BOTH perturbations (one alone misses problems that only move one way).
        _, res2 = pool.run(perturb=1)
        _, res3 = pool.run(perturb=-1)
    finally:
        pool.close()
    st_ref = np.array([r[1] for r in res]); x_ref = np.array([r[4] for r in res])
    st2 = np.array([r[1] for r in res2]); x2 = np.array([r[4] for r in res2])
    st3 = np.array([r[1] for r in res3]); x3 = np.array([r[4] for r in res3])
    k = L.ia + 1
    out = {"cpu_baseline": {"value": sample / dt, "unit": UNIT, "cores": pool.cores, "kind": cpu_kind_label(pool.kind),
                            "native": "reference C++ (oracle/_ref)" if pool.kind == "ref" else "plain-C oracle",
                            "sample": "first %d problems of the same batch, scipy SLSQP with 2-point finite differences on the "
                                      "reference's closures, one process per core (%d); closures built before the clock" % (sample, pool.cores),
                            "seconds": dt, "status_histogram": hist(st_ref)}}
    d2 = np.abs(x2[:, :k] - x_ref[:, :k]).max(1); d3 = np.abs(x3[:, :k] - x_ref[:, :k]).max(1)
    all0 = (st_ref == 0) & (st2 == 0) & (st3 == 0)
    stable = all0 & (d2 <= 1e-5) & (d3 <= 1e-5)
    same_self = (st_ref == st2) & (st_ref == st3)

    def agreement(xg, sg, mode):
        dcp = np.abs(xg[:, :k] - x_ref[:, :k]).max(1)
        both = (st_ref == 0) & (sg == 0)
        return {"jacobian": mode, "problems": int(sample), "reference_status0": int((st_ref == 0).sum()),
                "both_status0": int(both.sum()), "same_success_flag": int(((st_ref == 0) == (sg == 0)).sum()),
                "same_status": int((st_ref == sg).sum()),
                "same_status_where_reference_agrees_with_itself": int(((st_ref == sg) & same_self).sum()),
                "status0_within_1e-5": int((dcp[both] <= 1e-5).sum()),
                "status0_within_1e-3": int((dcp[both] <= 1e-3).sum()),
                "reference_stable_problems": int(stable.sum()),
                "reference_stable_within_1e-5": int((dcp[stable & (sg == 0)] <= 1e-5).sum())}
    out["parity_sample"] = [agreement(arrays["x"][:sample], arrays["status"][:sample], jacobian)]
    if "other_x" in arrays:
        out["parity_sample"].append(agreement(arrays["other_x"][:sample], arrays["other_status"][:sample], arrays["other"]))
    out["reference_self_consistency"] = {
        "perturbation": "x0 + 1 ulp and x0 - 1 ulp", "problems": int(sample), "all_status0": int(all0.sum()),
        "same_status": int(same_self.sum()), "status0_within_1e-5": int(stable.sum()),
        "status0_within_1e-3": int((all0 & (d2 <= 1e-3) & (d3 <= 1e-3)).sum())}
    return out


def bench_c5_strong(G, steps, warmup):
    """BASELINE configs[4]: 1,048,576 bicycle / unicycle problems IN TOTAL (half angular-rate, half curvature bound),
    replicated on every rank's host and sharded over the ranks by distributed.solve_sharded -- the product's own
    shard + all-gather route (strong scaling: the total is fixed as N grows)."""
    from trajectory_generator_b200 import distributed as tgd, synthetic
    halves = [synthetic.make_c5(C5_TOTAL // 2, kind) for kind in ("angular_rate", "curvature")]
    times, outs = [], None
    for it in range(warmup + steps):
        G.barrier()
        t = time.perf_counter()
        outs = [tgd.solve_sharded(b.spec, b.par, b.x0, jacobian=G.args.jacobian) for b in halves]
        G.barrier()
        if it >= warmup:
            times.append(time.perf_counter() - t)
    sec = G.max_over_ranks(float(np.mean(times)))
    st = np.concatenate([o["status"] for o in outs]); nit = np.concatenate([o["nit"] for o in outs])
    Ls = [b.layout for b in halves]
    return {"metric": METRIC, "value": C5_TOTAL / sec, "unit": UNIT, "ms_per_step": sec * 1e3, "steps": steps, "warmup": warmup,
            "scaling": "strong", "timing": "wall clock between barriers (max over ranks): host buffers in, host rows out",
            "config": {"workload": "bicycle/unicycle kinematic trajectories with angular-rate / curvature + acceleration bounds, "
                                   "%d problems in total over %d GPU(s)" % (C5_TOTAL, G.world),
                       "config": "C5", "total_problems": C5_TOTAL, "api": "distributed.solve_sharded (shard -> tg_solve_batch -> one all-gather of result rows)"},
            "shape": {"d": Ls[0].d, "N": Ls[0].N, "n": Ls[0].n, "m": Ls[0].m, "meq": Ls[0].meq},
            "solve_stats": {"mean_nit": float(nit.mean()), "max_nit": int(nit.max()), "status_histogram": hist(st)},
            "e2e": {"value": C5_TOTAL / sec, "unit": UNIT,
                    "h2d_bytes_per_step": int(sum(8 * (C5_TOTAL // 2 // G.world) * (l.P + l.n) for l in Ls)),
                    "d2h_bytes_per_step": int(sum(8 * (C5_TOTAL // 2) * (l.n + 4) for l in Ls)),
                    "api": "distributed.solve_sharded"}}


def bench_c1_latency(G):
    """BASELINE configs[0]: the single problem of test_2D_trajectory.py through the drop-in class -- latency of one
    generate_trajectory call (packing, H2D, solve, D2H)."""
    from trajectory_generator_b200 import synthetic
    from trajectory_generator_b200.trajectory_generator import TrajectoryGenerator
    d, cc, kw = synthetic.c1_problem()
    gen = TrajectoryGenerator(d)
    ts = []
    for it in range(8):
        t = time.perf_counter()
        gen.generate_trajectory(cc, **kw)
        if it >= 3:
            ts.append(time.perf_counter() - t)
    r = gen.last_result
    rec = {"metric": "single_problem_latency", "value": float(np.median(ts)) * 1e3, "unit": "ms", "higher_is_better": False,
           "config": {"workload": "test_2D_trajectory.py: single 2D order-3 B-spline, 3 corridors, start/end waypoints with velocity",
                      "config": "C1", "api": "TrajectoryGenerator(2).generate_trajectory(container, 'minimal_time_path', 10)"},
           "status": int(r.status), "nit": int(r.nit), "calls": len(ts)}
    return rec, (d, cc, kw, r)


def c1_cpu(d, cc, kw, r):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import tg_oracle
    op = tg_oracle.OracleProblem(d, cc, kw["objective_function_type"], kw["num_intervals_free_space"],
                                 native_kind=cpu_path_available())
    op.solve()
    t = time.perf_counter()
    res = op.solve()
    dt = time.perf_counter() - t
    k = 2 * op.N + 1
    return {"cpu_baseline": {"value": dt * 1e3, "unit": "ms", "cores": 1, "kind": "port",
                             "sample": "the same problem, scipy SLSQP on the reference's closures, one core"},
            "parity": {"reference_status": int(res.status), "reference_nit": int(res.nit), "status": int(r.status), "nit": int(r.nit),
                       "max_abs_dcp": float(np.abs(np.asarray(r.x)[:k] - res.x[:k]).max())}}


def main():
    args = parse()
    out_stream = _claim_stdout()
    rank = int(os.environ.get("RANK", "0"))
    if args.impl == "reference":
        if rank == 0:
            reference_arm(args, out_stream)
        return
    import torch
    if not torch.cuda.is_available():
        # a driver that is momentarily busy (seen once right after another process exited) answers "initialization
        # failed": wait and start over in a fresh process a few times before giving up
        tries = int(os.environ.get("TG_BENCH_CUDA_RETRY", "0"))
        if tries < 4:
            time.sleep(5 + 5 * tries)
            os.environ["TG_BENCH_CUDA_RETRY"] = str(tries + 1)
            os.dup2(out_stream.fileno(), 1)
            os.execv(sys.executable, [sys.executable] + sys.argv)
        raise SystemExit("bench.py: no CUDA device (the product has no CPU path; use --impl reference for the CPU arm)")
    from trajectory_generator_b200 import synthetic
    G = Gpu(args)
    name = args.config
    B = args.batch or synthetic.FULL_BATCH[name]
    cores = os.cpu_count() or 1
    sampler = ClockSampler(G.local)
    if G.rank == 0:
        sampler.start()
    head, arrays = bench_config(G, name, B, args.steps, args.warmup, full=True)
    if G.rank == 0:
        sampler.stop_flag = True
        sampler.join(timeout=2)
    line = {"metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": G.world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic"}
    for k in ("config", "shape", "solve_stats", "roofline", "e2e", "evals", "sampling", "gpu_launches"):
        line[k] = head[k]
    for k in head:
        if k.endswith("_mode"):
            line[k] = head[k]
    line["schedule"] = "fused persistent kernel" if args.fused else "lock-step stage kernels"
    line["clocks"] = sampler.summary()
    do_cpu = G.world == 1 and not args.no_cpu_baseline and cpu_path_available()
    if do_cpu:
        try:
            line.update(parity_against_cpu(name, arrays, args.cpu_sample or default_cpu_sample(name, cores), cores, args.jacobian))
        except Exception as exc:      # the baseline is reported, never required
            line["cpu_baseline"] = {"error": repr(exc)}
    del arrays
    torch.cuda.empty_cache()

    # ---- the other BASELINE configurations
    if not args.quick:
        subs = {}
        sub_steps, sub_warm = min(args.steps, 2), min(args.warmup, 3)
        if G.world == 1:
            try:
                rec, c1 = bench_c1_latency(G)
                if do_cpu:
                    rec.update(c1_cpu(*c1))
                subs["C1"] = rec
            except Exception as exc:
                subs["C1"] = {"error": repr(exc)}
            for sub in ("C2", "C3", "C4"):
                if sub == name:
                    continue
                try:
                    rec, arr = bench_config(G, sub, synthetic.FULL_BATCH[sub], sub_steps, sub_warm, full=False)
                    if do_cpu:
                        rec.update(parity_against_cpu(sub, arr, args.cpu_sample or default_cpu_sample(sub, cores), cores, args.jacobian))
                    subs[sub] = rec
                    del arr
                    torch.cuda.empty_cache()
                except Exception as exc:
                    subs[sub] = {"error": repr(exc)}
        try:
            subs["C5"] = bench_c5_strong(G, sub_steps, 1)
        except Exception as exc:
            subs["C5"] = {"error": repr(exc)}
        # ---- f3: problems of different shapes in ONE call (tg_solve_mixed_host) against bucket-by-bucket calls; shapes
        #      chosen from raw geometry on the device (f2 -> f3); the drop-in class on a list of containers
        if G.world == 1:
            for key, fn in (("mixed_shapes", bench_mixed), ("shapes_from_geometry", bench_geometry), ("dropin_e2e", bench_dropin)):
                try:
                    subs[key] = fn(G)
                except Exception as exc:
                    subs[key] = {"error": repr(exc)}
        line["configs"] = subs
    if G.rank == 0:
        print(json.dumps(line), file=out_stream, flush=True)
    if G.world > 1:
        G.dist.destroy_process_group()


def bench_mixed(G):
    from trajectory_generator_b200 import batch as tgb, synthetic
    MB = 4096
    gens = (("C2", synthetic.make_c2, 2), ("C3", synthetic.make_c3, 3), ("C4", synthetic.make_c4, 4))
    mbs = [g(MB, seed=synthetic.SEED0 + k + 100 * r) for _, g, k in gens for r in (1, 2)]
    mbs += [synthetic.make_c5(MB, kind, seed=synthetic.SEED0 + 5 + 100) for kind in ("angular_rate", "curvature")]
    buckets = [(b.spec, b.par, b.x0) for b in mbs]
    jac = G.args.jacobian
    runs = {"bucket_by_bucket": lambda: [tgb.solve_host(sp_, p_, x_, jacobian=jac) for sp_, p_, x_ in buckets],
            "one_call": lambda: tgb.solve_mixed_host(buckets, jacobian=jac)}
    tm, res_m = {}, {}
    for label, fn in runs.items():
        fn()
        ts = []
        for _ in range(2):
            t = time.perf_counter(); res_m[label] = fn(); ts.append(time.perf_counter() - t)
        tm[label] = min(ts)
    same = all(np.array_equal(a["x"], b["x"]) and np.array_equal(a["status"], b["status"])
               for a, b in zip(res_m["bucket_by_bucket"], res_m["one_call"]))
    return {"workload": "%d buckets of %d problems: C2, C3, C4 (two seeds each), C5a, C5c" % (len(buckets), MB),
            "problems": MB * len(buckets), "unit": UNIT, "api": "tg_solve_mixed_host (C-ABI, host buffers)",
            "one_call": MB * len(buckets) / tm["one_call"], "bucket_by_bucket": MB * len(buckets) / tm["bucket_by_bucket"],
            "identical_results": bool(same)}


def bench_geometry(G):
    """Raw 3-D corridor polylines in (segment lengths 5 .. 11.5: 2 .. 3 intervals per corridor by the reference's rule),
    shapes chosen on the device, boxes / parameter rows / initial guesses built on the device, one solve call."""
    torch = G.torch
    from trajectory_generator_b200.batched import CorridorProblems
    rng = np.random.default_rng(20261018)
    B, ncorr = 32768, 3
    pts = np.zeros((B, 3, ncorr + 1))
    pts[:, :, 0] = rng.uniform(-5, 5, (B, 3))
    direction = rng.normal(size=(B, 3)); direction /= np.linalg.norm(direction, 2, 1)[:, None]
    for i in range(1, ncorr + 1):
        direction = direction + rng.normal(size=(B, 3)) * 0.35
        direction /= np.linalg.norm(direction, 2, 1)[:, None]
        pts[:, :, i] = pts[:, :, i - 1] + direction * rng.uniform(5, 11.5, B)[:, None]
    pads = np.stack([rng.uniform(2, 3, (B, ncorr)), rng.uniform(2, 3, (B, ncorr)), rng.uniform(2, 4, (B, ncorr))], 2)
    v0 = pts[:, :, 1] - pts[:, :, 0]; v0 /= np.linalg.norm(v0, 2, 1)[:, None]
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(G.dev)
    tp, tpad, tv = t(pts), t(pads), t(v0)
    ts = []
    for it in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        cp = CorridorProblems(3, corridor_points=tp, corridor_pads=tpad, start_velocity=tv, end_zero_velocity=True,
                              max_velocity=5.0, max_acceleration=0.3, objective_function_type="minimal_velocity_path")
        out = cp.solve(jacobian=G.args.jacobian)
        torch.cuda.synchronize()
        if it:
            ts.append(time.perf_counter() - t0)
    shapes = cp.shapes()
    return {"workload": "%d raw 3-D corridor polylines (3 corridors, segment lengths 5 .. 11.5), shapes from geometry" % B,
            "problems": B, "shapes": len(shapes), "largest_shape": max(c for _, c in shapes), "unit": UNIT,
            "api": "batched.CorridorProblems (tg_sfc_intervals_batch -> sort by shape key -> BatchedProblem per shape -> tg_solve_mixed_batch)",
            "value": B / min(ts), "includes": "interval rule, grouping, corridor boxes, parameter rows, initial guesses and the solve, device tensors in / out",
            "status0_fraction": float((out["status"] == 0).double().mean().item())}


def bench_dropin(G):
    """The drop-in class on a list of containers: TrajectoryGenerator.generate_trajectories(list) -- vectorised packing
    (problem.pack_problems), H2D, solve, D2H, result objects.  Containers are built outside the clock."""
    from trajectory_generator_b200 import synthetic
    from trajectory_generator_b200.trajectory_generator import TrajectoryGenerator
    from trajectory_generator_b200.problem import pack_problems
    rec = {"unit": "containers/s", "api": "TrajectoryGenerator(d).generate_trajectories(list_of_containers)", "configs": {}}
    for name, count in (("C2", 16384), ("C4", 8192)):
        bt = synthetic.make(name, count)
        items = [synthetic.container_for(bt, i) for i in range(count)]
        d, kw = items[0][0], items[0][2]
        ccs = [c[1] for c in items]
        gen = TrajectoryGenerator(d)
        ts = []
        for it in range(3):
            t0 = time.perf_counter()
            res = gen.generate_trajectories(ccs, **kw)
            if it:
                ts.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        pack_problems(d, ccs, kw.get("objective_function_type", "minimal_velocity_and_time_path"), kw.get("num_intervals_free_space"))
        tp = time.perf_counter() - t0
        rec["configs"][name] = {"containers": count, "value": count / min(ts), "packing_only": count / tp,
                                "status0_fraction": float(np.mean([r.status == 0 for r in res]))}
    rec["value"] = rec["configs"]["C2"]["value"]
    return rec


if __name__ == "__main__":
    main()
