"""Solve rate of shapes whose QP scratch does not fit in shared memory (workspace slots), and the cost of that placement
on shapes that fit.
usage: large_shapes_bench.py OUTDIR [--reps R]
  * corridors8_3d and waypoints3d (tests/test_large_shapes.py) as batches of perturbed copies, 4,096 and 16,384
    problems, fd mode, maxiter 500: trajectories/s (CUDA events around the solve, inputs resident), the line-search / QP
    split (tg_set_stage_timing), the status histogram, the bytes of the workspace slots against the 126 MB L2;
  * TG_QP_FAR=1 against the default placement on C2 and C4 at 65,536 problems, alternated in one run (plus the
    default placement with the far kernel's 64 lanes, TG_QP_GS=64, to separate lanes from placement).
Writes OUTDIR/large_shapes_bench.json with the GPU's name and power limit."""
import argparse, ctypes, json, os, subprocess, sys
import numpy as np
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
from trajectory_generator_b200 import batch as tgb, synthetic as syn, _native
import test_large_shapes as large

ap = argparse.ArgumentParser()
ap.add_argument("outdir")
ap.add_argument("--reps", type=int, default=2)
args = ap.parse_args()
os.makedirs(args.outdir, exist_ok=True)
dev = torch.device("cuda:0")
lib = _native.lib()
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip()
res = dict(gpu=gpu, shapes=[], placement=[])


def run(spec, par, x0, maxiter, mode, reps):
    """mean / min ms of `reps` timed solves after one warm-up, then one solve with stage timing"""
    bufs = tgb.SolveBuffers(spec, par.shape[0], dev)
    ts = []
    for r in range(reps + 1):
        x = x0.clone()
        s = torch.cuda.Event(enable_timing=True); e = torch.cuda.Event(enable_timing=True)
        s.record(); out = tgb.solve(spec, par, x, maxiter=maxiter, jacobian=mode, buffers=bufs); e.record()
        torch.cuda.synchronize()
        if r:
            ts.append(s.elapsed_time(e))
    lib.tg_set_stage_timing(1)
    x = x0.clone(); tgb.solve(spec, par, x, maxiter=maxiter, jacobian=mode, buffers=bufs); torch.cuda.synchronize()
    lib.tg_set_stage_timing(0)
    st = (ctypes.c_double * 6)(); lib.tg_last_solve_stats(st, 6)
    return ts, st, out, bufs


for name in ("corridors8_3d", "waypoints3d"):
    spec, par_all, x_all = large._perturbed(name, 16384, seed=1)
    for B in (4096, 16384):
        par = torch.from_numpy(par_all[:B]).to(dev); x0 = torch.from_numpy(x_all[:B]).to(dev)
        ts, st, out, bufs = run(spec, par, x0, 500, "fd", args.reps)
        plan = tgb.solve_plan(spec, B)
        status, counts = np.unique(out["status"].cpu().numpy(), return_counts=True)
        row = dict(shape=name, B=B, n=int(x0.shape[1]), ms=ts, traj_per_s=B / min(ts) * 1e3, ms_ls=st[0], ms_qp=st[1],
                   rounds=int(st[5]), status={int(k): int(v) for k, v in zip(status, counts)},
                   nit_mean=out["nit"].float().mean().item(), plan=plan, slot_bytes=plan["slot_kib"] * 1024,
                   slots_over_l2=plan["slot_kib"] * 1024 / 126e6, workspace_bytes=int(bufs.ws.numel()))
        print(json.dumps(row), flush=True)
        res["shapes"].append(row)

arms = [("default", {}), ("TG_QP_GS=64", {"TG_QP_GS": "64"}), ("TG_QP_FAR=1", {"TG_QP_FAR": "1"})]
for name in ("C2", "C4"):
    b = syn.make(name, 65536)
    par = torch.from_numpy(b.par).to(dev); x0 = torch.from_numpy(b.x0).to(dev)
    for rnd in range(2):               # alternated: default, lanes only, far, default, ...
        for label, env in arms:
            os.environ.update(env)
            ts, st, out, _ = run(b.spec, par, x0, 100, "fd", args.reps)
            row = dict(config=name, arm=label, round=rnd, B=65536, ms=ts, traj_per_s=65536 / min(ts) * 1e3, ms_ls=st[0],
                       ms_qp=st[1], status0=(out["status"] == 0).float().mean().item(),
                       xsum=out["x"].double().sum().item(), plan=tgb.solve_plan(b.spec, 65536))
            for k in env:
                os.environ.pop(k)
            print(json.dumps(row), flush=True)
            res["placement"].append(row)

with open(os.path.join(args.outdir, "large_shapes_bench.json"), "w") as f:
    json.dump(res, f, indent=1)
