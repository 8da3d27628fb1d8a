"""What the post-solve polish (batch.polish; DESIGN.md §4 *Polish*) buys and costs, next to the obvious workaround of a
plain solve with a tighter tolerance.

    python scripts/polish_bench.py OUTDIR [--b 65536] [--b-c5a 16384] [--repeats 2]

C2, C3 and C4 x b and C5a x b-c5a, in analytic and fd modes.  Per configuration, alternated `repeats` times after an
untimed warm-up of each: the solve with multipliers, the polish of a copy of its result, and the baseline, a plain solve
at ftol = 1e-10, maxiter = 400 with multipliers; device time from CUDA events around each call.  Reported: the status-0
share; over the status-0 problems the stationarity (kkt[0]) median / p99 and the shares <= 1e-6 and <= 1e-8 before and
after the polish and of the baseline; the polish_status histogram; over the replaced rows the mean change of f and of
the maximum violation (kkt[1]); a SHA-256 checksum of the polished outputs (x, f, violation, lam, kkt, polish_status,
polish_iters), which compares the polish's bits across versions.  Writes OUTDIR/polish.json and OUTDIR/polish.md with the card's name and power limit
read in the same run."""
import argparse
import hashlib
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def _timed(fn):
    import torch
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    torch.cuda.synchronize()
    ev[0].record()
    out = fn()
    ev[1].record()
    torch.cuda.synchronize()
    return out, ev[0].elapsed_time(ev[1])


def _stationarity(kkt, ok):
    s = kkt[ok, 0]
    if s.size == 0:
        return dict(median=float("nan"), p99=float("nan"), le_1e6=0.0, le_1e8=0.0)
    return dict(median=float(np.median(s)), p99=float(np.percentile(s, 99)), le_1e6=float(np.mean(s <= 1e-6)),
                le_1e8=float(np.mean(s <= 1e-8)))


def run(bt, jac, repeats):
    import torch

    from trajectory_generator_b200 import batch
    par, x0 = torch.from_numpy(bt.par).cuda(), torch.from_numpy(bt.x0).cuda()
    solve = lambda: batch.solve(bt.spec, par, x0.clone(), jacobian=jac, multipliers=True)
    base = lambda: batch.solve(bt.spec, par, x0.clone(), jacobian=jac, multipliers=True, ftol=1e-10, maxiter=400)

    def polish(sol):
        rows = {k: sol[k].clone() for k in ("x", "f", "status", "violation", "lam", "kkt")}
        return _timed(lambda: batch.polish(bt.spec, par, rows))

    sol = solve(); polish(sol); base()                 # warm-up: module loads, allocator
    t = dict(solve=[], polish=[], baseline=[])
    for _ in range(repeats):
        sol, ms = _timed(solve); t["solve"].append(ms)
        pol, ms = polish(sol); t["polish"].append(ms)
        bl, ms = _timed(base); t["baseline"].append(ms)
    sol = {k: v.cpu().numpy() for k, v in sol.items()}
    pol = {k: v.cpu().numpy() for k, v in pol.items()}
    bl = {k: v.cpu().numpy() for k, v in bl.items()}
    ok, okb = sol["status"] == 0, bl["status"] == 0
    rep = ok & (pol["polish_status"] <= 1)
    ck = hashlib.sha256()
    for k in ("x", "f", "violation", "lam", "kkt", "polish_status", "polish_iters"):
        ck.update(np.ascontiguousarray(pol[k]).tobytes())
    hist = {batch.POLISH_STATUS[k]: int(np.sum(pol["polish_status"][ok] == k)) for k in range(6) if k != 4}
    return dict(status0=float(ok.mean()), before=_stationarity(sol["kkt"], ok), after=_stationarity(pol["kkt"], ok),
                polish_status=hist, replaced=int(rep.sum()),
                mean_df=float(np.mean(pol["f"][rep] - sol["f"][rep])) if rep.any() else 0.0,
                mean_dviol=float(np.mean(pol["kkt"][rep, 1] - sol["kkt"][rep, 1])) if rep.any() else 0.0,
                baseline_status0=float(okb.mean()), baseline=_stationarity(bl["kkt"], okb),
                checksum=ck.hexdigest(), ms=t)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir")
    ap.add_argument("--b", type=int, default=65536)
    ap.add_argument("--b-c5a", type=int, default=16384)
    ap.add_argument("--repeats", type=int, default=2)
    a = ap.parse_args()
    import torch

    from multistart_bench import card
    from trajectory_generator_b200 import synthetic
    if not torch.cuda.is_available():
        raise SystemExit("polish_bench.py needs a CUDA device")
    os.makedirs(a.outdir, exist_ok=True)
    name, power = card()
    rows = []
    for jac in ("analytic", "fd"):
        for cfg in ("C2", "C3", "C4", "C5a"):
            B = a.b_c5a if cfg == "C5a" else a.b
            r = dict(config=cfg, B=B, jacobian=jac, card=name, power_limit=power, **run(synthetic.make(cfg, B), jac, a.repeats))
            rows.append(r)
            print(json.dumps(r), flush=True)
    with open(os.path.join(a.outdir, "polish.json"), "w") as fh:
        json.dump(dict(rows=rows, card=name, power_limit=power), fh, indent=1)
    st = lambda s: "%.1e / %.1e | %.2f / %.2f" % (s["median"], s["p99"], 100 * s["le_1e6"], 100 * s["le_1e8"])
    lines = ["%s, power limit %s" % (name, power), "",
             "| jacobian | config | B | status 0 % | stationarity before: median / p99 \\| % <= 1e-6 / 1e-8 "
             "| after polish | polished / improved / rejected / degenerate / nonfinite | mean df | mean d max viol "
             "| ftol=1e-10, maxiter=400: status 0 % \\| median / p99 \\| % <= 1e-6 / 1e-8 "
             "| ms solve / polish / low-ftol solve |",
             "|---|---|---|---|---|---|---|---|---|---|---|"]
    for r in rows:
        h = r["polish_status"]
        med = lambda v: float(np.median(v))
        lines.append("| %s | %s | %d | %.1f | %s | %s | %s | %.2e | %.2e | %.1f \\| %s | %.0f / %.0f / %.0f |" % (
            r["jacobian"], r["config"], r["B"], 100 * r["status0"], st(r["before"]), st(r["after"]),
            " / ".join(str(h[k]) for k in ("polished", "improved", "rejected", "degenerate", "nonfinite")),
            r["mean_df"], r["mean_dviol"], 100 * r["baseline_status0"], st(r["baseline"]),
            med(r["ms"]["solve"]), med(r["ms"]["polish"]), med(r["ms"]["baseline"])))
    with open(os.path.join(a.outdir, "polish.md"), "w") as fh:
        fh.write("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
