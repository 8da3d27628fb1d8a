"""Multi-start solves (batch.solve_multistart) on the synthetic configurations: how much K seeded starts per problem buy
and what they cost.

    python scripts/multistart_bench.py OUTDIR [--c2 65536] [--c4 65536] [--c5 16384] [--starts 1,2,4,8]
                                              [--spreads 0.05,0.1,0.25] [--jacobian analytic]

For every configuration, K and spread: the fraction of problems with status 0 and the fraction converged and feasible
at batch.MULTISTART_TOL (true maximum violation), the mean f against K = 1 over the problems that converged in both,
problems/s (B problems, not B * K rows) and the device time of expand / solve / select from CUDA events (one run per
point after an untimed warm-up solve of each configuration).  Writes OUTDIR/multistart.json and OUTDIR/multistart.md
with the card's name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    import torch
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return name, q


def run_point(bt, K, spread, jacobian, seed=0):
    import torch

    from trajectory_generator_b200 import batch
    par, x0 = torch.from_numpy(bt.par).cuda(), torch.from_numpy(bt.x0).cuda()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    torch.cuda.synchronize()
    ev[0].record()
    par_e, x_e = batch.multistart_expand(bt.spec, par, x0, K, seed, spread)
    ev[1].record()
    sol = batch.solve(bt.spec, par_e, x_e, jacobian=jacobian)
    ev[2].record()
    sel = batch.multistart_select(bt.spec, par, sol, K)
    ev[3].record()
    torch.cuda.synchronize()
    ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(3)]
    out = {k: sel[k].cpu().numpy() for k in ("f", "status", "max_violation", "best_start")}
    return out, ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir")
    ap.add_argument("--c2", type=int, default=65536)
    ap.add_argument("--c4", type=int, default=65536)
    ap.add_argument("--c5", type=int, default=16384, help="C5a (bicycle, angular-rate bound) sample size")
    ap.add_argument("--starts", default="1,2,4,8")
    ap.add_argument("--spreads", default="0.05,0.1,0.25")
    ap.add_argument("--jacobian", default="analytic", choices=("analytic", "fd"))
    a = ap.parse_args()
    import torch

    from trajectory_generator_b200 import batch, synthetic
    if not torch.cuda.is_available():
        raise SystemExit("multistart_bench.py needs a CUDA device")
    os.makedirs(a.outdir, exist_ok=True)
    name, power = card()
    starts = [int(v) for v in a.starts.split(",")]
    spreads = [float(v) for v in a.spreads.split(",")]
    tol = batch.MULTISTART_TOL
    rows = []
    for cfg, B in (("C2", a.c2), ("C4", a.c4), ("C5a", a.c5)):
        if B <= 0:
            continue
        bt = synthetic.make(cfg, B)
        run_point(bt, 1, 0.0, a.jacobian)          # warm-up: module loads, allocator
        base = None
        for K in starts:
            for spread in (spreads if K > 1 else [0.0]):
                out, ms = run_point(bt, K, spread, a.jacobian)
                if K == 1:
                    base = out
                ok = (out["status"] == 0) & (out["max_violation"] <= tol)
                r = dict(config=cfg, B=B, K=K, spread=spread, jacobian=a.jacobian,
                         status0=float(np.mean(out["status"] == 0)), feasible=float(np.mean(ok)),
                         ms_expand=ms[0], ms_solve=ms[1], ms_select=ms[2], problems_per_s=B / (sum(ms) * 1e-3),
                         won_by_start0=float(np.mean(out["best_start"] == 0)), card=name, power_limit=power)
                if base is not None:
                    both = (base["status"] == 0) & (out["status"] == 0)
                    r["both_converged"] = int(both.sum())
                    r["mean_f_K1"] = float(base["f"][both].mean()) if both.any() else float("nan")
                    r["mean_f"] = float(out["f"][both].mean()) if both.any() else float("nan")
                rows.append(r)
                print(json.dumps(r), flush=True)
    with open(os.path.join(a.outdir, "multistart.json"), "w") as fh:
        json.dump(rows, fh, indent=1)
    lines = ["%s, power limit %s, jacobian=%s, tol=%g" % (name, power, a.jacobian, tol), "",
             "| config | B | K | spread | status 0 | conv. + feasible | mean f (K=1) on both conv. | problems/s | "
             "expand / solve / select ms |", "|---|---|---|---|---|---|---|---|---|"]
    for r in rows:
        lines.append("| %s | %d | %d | %g | %.4f | %.4f | %.6g (%.6g) | %.0f | %.2f / %.1f / %.2f |" % (
            r["config"], r["B"], r["K"], r["spread"], r["status0"], r["feasible"], r.get("mean_f", float("nan")),
            r.get("mean_f_K1", float("nan")), r["problems_per_s"], r["ms_expand"], r["ms_solve"], r["ms_select"]))
    with open(os.path.join(a.outdir, "multistart.md"), "w") as fh:
        fh.write("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
