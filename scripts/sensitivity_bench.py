"""What the parameter sensitivities (batch.sensitivity; DESIGN.md §4 *Sensitivities*) cost and how accurate they are.

    python scripts/sensitivity_bench.py OUTDIR [--b 65536] [--b-c5a 16384] [--repeats 2] [--check 256]

C2, C3 and C4 x b and C5a x b-c5a, in analytic and fd solve modes.  Per configuration, alternated `repeats` times after
an untimed warm-up of each: the solve with multipliers, the polish of a copy of its result, and the sensitivities of the
polished result for random upstream gradients x_bar, f_bar; device time from CUDA events around each call.  Reported:
the sens_status histogram, and the re-solve accuracy on the first `check` problems: for a random direction delta over
the parameter row, <par_bar, delta> against (loss(x+) - loss(x-)) / 2h, x+- re-solved from x* at par +- h delta
(h = 1e-5, ftol = 1e-12, maxiter = 400, polished, then polished again at tol 1e-12), over the rows whose sens_status
is ok and whose two re-solves are stationary to 1e-11 with the solve's working set and bound pattern.  Writes OUTDIR/sensitivity.json
and OUTDIR/sensitivity.md with the card's name and power limit read in the same run."""
import argparse
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


def _accuracy(bt, jac, sol, x_bar, f_bar, sens, count, h=1e-5):
    """relative errors of <par_bar, delta> against re-solves on the first `count` rows (see the top of the file)"""
    import torch

    from trajectory_generator_b200 import batch
    L = bt.layout
    rows = slice(0, count)
    rng = np.random.default_rng(17)
    par = bt.par[rows]
    delta = rng.standard_normal(par.shape) * np.maximum(1.0, np.abs(par))
    x_star = sol["x"][rows].contiguous()
    lam = sol["lam"][rows].cpu().numpy()
    W = (np.arange(L.m)[None] < L.meq) | (lam > 0)
    xl = np.full(L.n, -np.inf); xu = np.full(L.n, np.inf)
    xl[L.ia:L.it0] = 10e-8
    if L.it0 < L.n:
        xl[L.it0:] = 0; xu[L.it0:] = L.N - 3
    at_bound = lambda x: (x == xl) | (x == xu)
    bnd = at_bound(x_star.cpu().numpy())
    keep = (sens["sens_status"][rows].cpu().numpy() == 0) & (sol["status"][rows].cpu().numpy() == 0)
    res = []
    for s in (1, -1):
        # a second polish at tol 1e-12: the default 1e-8 leaves errors of x that the 1 / 2h below would amplify; rows
        # count when stationary to 1e-11 max(1, max|g|) (the `inexact` test of the sensitivities at tol 1e-11)
        P = torch.from_numpy(par + s * h * delta).cuda()
        r = batch.solve(bt.spec, P, x_star.clone(), jacobian=jac, ftol=1e-12, maxiter=400, polish=True)
        batch.polish(bt.spec, P, r, maxiter=20, tol=1e-12)
        tight = batch.sensitivity(bt.spec, P, r, torch.zeros_like(r["x"]), tol=1e-11)["sens_status"].cpu().numpy() <= 1
        r = {k: v.cpu().numpy() for k, v in r.items()}
        keep &= (r["status"] == 0) & tight & (((np.arange(L.m)[None] < L.meq) | (r["lam"] > 0)) == W).all(1)
        keep &= (at_bound(r["x"]) == bnd).all(1)
        res.append(r)
    xb, fb = x_bar[rows].cpu().numpy(), f_bar[rows].cpu().numpy()
    fd = (np.einsum("bn,bn->b", xb, res[0]["x"] - res[1]["x"]) + fb * (res[0]["f"] - res[1]["f"])) / (2 * h)
    an = np.einsum("bp,bp->b", sens["par_bar"][rows].cpu().numpy(), delta)
    err = np.abs(fd - an)[keep] / np.maximum(np.maximum(np.abs(fd), np.abs(an)), 1e-300)[keep]
    return dict(rows=count, compared=int(keep.sum()),
                median_rel_err=float(np.median(err)) if err.size else float("nan"),
                max_rel_err=float(err.max()) if err.size else float("nan"),
                within_1e4=int((err <= 1e-4).sum()))


def run(bt, jac, repeats, check):
    import torch

    from trajectory_generator_b200 import batch
    par, x0 = torch.from_numpy(bt.par).cuda(), torch.from_numpy(bt.x0).cuda()
    B, L = bt.par.shape[0], bt.layout
    g = torch.Generator(device="cuda").manual_seed(3)
    x_bar = torch.randn((B, L.n), dtype=torch.float64, device="cuda", generator=g)
    f_bar = torch.randn(B, dtype=torch.float64, device="cuda", generator=g)
    solve = lambda: batch.solve(bt.spec, par, x0.clone(), jacobian=jac, multipliers=True)

    def polish(sol):
        rows = {k: sol[k].clone() for k in ("x", "f", "status", "violation", "lam", "kkt")}
        return _timed(lambda: batch.polish(bt.spec, par, rows))

    sens = lambda pol: _timed(lambda: batch.sensitivity(bt.spec, par, pol, x_bar, f_bar))
    sol = solve(); pol, _ = polish(sol); sens(pol)          # warm-up: module loads, allocator
    t = dict(solve=[], polish=[], sensitivity=[])
    for _ in range(repeats):
        sol, ms = _timed(solve); t["solve"].append(ms)
        pol, ms = polish(sol); t["polish"].append(ms)
        out, ms = sens(pol); t["sensitivity"].append(ms)
    st = out["sens_status"].cpu().numpy()
    hist = {batch.SENS_STATUS[k]: int(np.sum(st == k)) for k in sorted(batch.SENS_STATUS)}
    return dict(sens_status=hist, accuracy=_accuracy(bt, jac, pol, x_bar, f_bar, out, min(check, B)), ms=t)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir")
    ap.add_argument("--b", type=int, default=65536)
    ap.add_argument("--b-c5a", type=int, default=16384)
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--check", type=int, default=256)
    a = ap.parse_args()
    import torch

    from multistart_bench import card
    from trajectory_generator_b200 import synthetic
    if not torch.cuda.is_available():
        raise SystemExit("sensitivity_bench.py needs a CUDA device")
    os.makedirs(a.outdir, exist_ok=True)
    name, power = card()
    rows = []
    for jac in ("analytic", "fd"):
        for cfg in ("C2", "C3", "C4", "C5a"):
            B = a.b_c5a if cfg == "C5a" else a.b
            r = dict(config=cfg, B=B, jacobian=jac, card=name, power_limit=power,
                     **run(synthetic.make(cfg, B), jac, a.repeats, a.check))
            rows.append(r)
            print(json.dumps(r), flush=True)
    with open(os.path.join(a.outdir, "sensitivity.json"), "w") as fh:
        json.dump(dict(rows=rows, card=name, power_limit=power), fh, indent=1)
    med = lambda v: float(np.median(v))
    lines = ["%s, power limit %s" % (name, power), "",
             "| jacobian | config | B | ok / nonstrict / inexact / degenerate / skipped / nonfinite / indefinite "
             "| re-solve check: compared of rows, within 1e-4, median / max rel. error | ms solve / polish / sensitivity |",
             "|---|---|---|---|---|---|"]
    for r in rows:
        h, acc = r["sens_status"], r["accuracy"]
        lines.append("| %s | %s | %d | %s | %d of %d, %d, %.1e / %.1e | %.0f / %.0f / %.0f |" % (
            r["jacobian"], r["config"], r["B"],
            " / ".join(str(h[k]) for k in ("ok", "nonstrict", "inexact", "degenerate", "skipped", "nonfinite",
                                            "indefinite")),
            acc["compared"], acc["rows"], acc["within_1e4"], acc["median_rel_err"], acc["max_rel_err"],
            med(r["ms"]["solve"]), med(r["ms"]["polish"]), med(r["ms"]["sensitivity"])))
    with open(os.path.join(a.outdir, "sensitivity.md"), "w") as fh:
        fh.write("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
