"""What batch.solve(..., multipliers=True) costs, and how stationary SLSQP's converged results are.

    python scripts/multipliers_bench.py OUTDIR [--b 65536] [--repeats 3]

Cost: C2 and C4 x B in finite-difference mode, solves with and without multipliers alternated (`repeats` pairs after an
untimed warm-up of each), device time from CUDA events; then one profiled run per configuration for the finish kernel's
time (torch.profiler, CUDA activities) with and without the multipliers.
Certificate: median and 99th percentile of each kkt entry (batch.KKT_FIELDS) over the status-0 problems of C2, C3, C4
and C5a x B, in both Jacobian modes.
Writes OUTDIR/multipliers.json and OUTDIR/multipliers.md with the card's name and power limit read in the same run."""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def timed_solve(bt, jacobian, multipliers):
    import torch

    from trajectory_generator_b200 import batch
    par, x0 = torch.from_numpy(bt.par).cuda(), torch.from_numpy(bt.x0).cuda()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    torch.cuda.synchronize()
    ev[0].record()
    out = batch.solve(bt.spec, par, x0, jacobian=jacobian, multipliers=multipliers)
    ev[1].record()
    torch.cuda.synchronize()
    return out, ev[0].elapsed_time(ev[1])


def finish_kernel_ms(bt, jacobian, multipliers):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        timed_solve(bt, jacobian, multipliers)
    return sum(e.device_time_total for e in prof.key_averages() if "tg_sqp_finish_kernel" in e.key) / 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir")
    ap.add_argument("--b", type=int, default=65536)
    ap.add_argument("--repeats", type=int, default=3)
    a = ap.parse_args()
    import torch

    from multistart_bench import card
    from trajectory_generator_b200 import batch, synthetic
    if not torch.cuda.is_available():
        raise SystemExit("multipliers_bench.py needs a CUDA device")
    os.makedirs(a.outdir, exist_ok=True)
    name, power = card()
    cost, cert = [], []
    for cfg in ("C2", "C4"):
        bt = synthetic.make(cfg, a.b)
        for mult in (False, True):
            timed_solve(bt, "fd", mult)                 # warm-up: module loads, allocator
        times = {False: [], True: []}
        for _ in range(a.repeats):
            for mult in (False, True):
                times[mult].append(timed_solve(bt, "fd", mult)[1])
        r = dict(config=cfg, B=a.b, jacobian="fd", ms_plain=times[False], ms_multipliers=times[True],
                 finish_ms_plain=finish_kernel_ms(bt, "fd", False), finish_ms_multipliers=finish_kernel_ms(bt, "fd", True),
                 card=name, power_limit=power)
        cost.append(r)
        print(json.dumps(r), flush=True)
    for jac in ("fd", "analytic"):
        for cfg in ("C2", "C3", "C4", "C5a"):
            bt = synthetic.make(cfg, a.b)
            out = {k: v.cpu().numpy() for k, v in timed_solve(bt, jac, True)[0].items()}
            ok = out["status"] == 0
            k = out["kkt"][ok]
            r = dict(config=cfg, B=a.b, jacobian=jac, status0=int(ok.sum()))
            for i, f in enumerate(batch.KKT_FIELDS):
                r[f] = dict(median=float(np.median(k[:, i])), p99=float(np.percentile(k[:, i], 99)))
            r["stationary_1e-6"] = float(np.mean(k[:, 0] <= 1e-6))
            r["stationary_1e-3"] = float(np.mean(k[:, 0] <= 1e-3))
            cert.append(r)
            print(json.dumps(r), flush=True)
    with open(os.path.join(a.outdir, "multipliers.json"), "w") as fh:
        json.dump(dict(cost=cost, certificate=cert, card=name, power_limit=power), fh, indent=1)
    lines = ["%s, power limit %s" % (name, power), "",
             "| config | B | solve ms, plain | solve ms, multipliers | finish kernel ms, plain / multipliers |",
             "|---|---|---|---|---|"]
    for r in cost:
        lines.append("| %s | %d | %s | %s | %.3f / %.3f |" % (
            r["config"], r["B"], " ".join("%.1f" % t for t in r["ms_plain"]),
            " ".join("%.1f" % t for t in r["ms_multipliers"]), r["finish_ms_plain"], r["finish_ms_multipliers"]))
    lines += ["", "| jacobian | config | status 0 | " + " | ".join("%s median / p99" % f for f in batch.KKT_FIELDS) +
              " | stationarity <= 1e-6 / 1e-3 |", "|---|---|---|---|---|---|---|---|"]
    for r in cert:
        lines.append("| %s | %s | %d | " % (r["jacobian"], r["config"], r["status0"]) +
                     " | ".join("%.2e / %.2e" % (r[f]["median"], r[f]["p99"]) for f in batch.KKT_FIELDS) +
                     " | %.3f / %.3f |" % (r["stationary_1e-6"], r["stationary_1e-3"]))
    with open(os.path.join(a.outdir, "multipliers.md"), "w") as fh:
        fh.write("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
