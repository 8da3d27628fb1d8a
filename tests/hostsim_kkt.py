"""TEST INFRASTRUCTURE: the host build of tests/hostsim/tg_hostsim_kkt.cpp (tg_hostsim.cpp plus tg_sqp_kkt) and scipy's
compiled SLSQP core driven the way hostsim_loader.scipy_core_solve drives it, keeping its multipliers.  The product
never loads either."""
import ctypes
import os
import subprocess

import numpy as np

import hostsim_loader
from hostsim_loader import ND, NI, CSRC, HERE

SRC = os.path.join(HERE, "hostsim", "tg_hostsim_kkt.cpp")


class HostSimKKT(hostsim_loader.HostSim):
    def solve_kkt(self, pp, maxiter=100, ftol=1e-6, fd=False):
        """solve plus the multipliers lam [m] and the KKT certificate kkt [4] of the final state (tg_sqp_kkt)"""
        L = pp.layout
        x = np.clip(pp.x0, pp.xl, pp.xu).copy()
        f = np.zeros(1); st = np.zeros(1, np.int32); nit = np.zeros(1, np.int32); nfev = np.zeros(1, np.int32)
        lam = np.zeros(max(L.m, 1)); kkt = np.zeros(4)
        self.lib.hs_solve_kkt.argtypes = [NI, ND, ND, ctypes.c_int, ctypes.c_double, ctypes.c_int, ND, NI, NI, NI, ND, ND]
        self.lib.hs_solve_kkt(pp.spec, pp.par, x, maxiter, ftol, 1 if fd else 0, f, st, nit, nfev, lam, kkt)
        return dict(x=x, f=f[0], status=int(st[0]), nit=int(nit[0]), nfev=int(nfev[0]), lam=lam[:L.m], kkt=kkt)


def load(tag="", flags=()):
    """The host build with the certificate; `flags` as in hostsim_loader.load_variant (-DTG_NO_ELIM, -DTG_FUSED_LM_FAR)."""
    out = os.path.join(HERE, "hostsim", "_build_hostsim_kkt%s.so" % ("_" + tag if tag else ""))
    deps = [SRC, hostsim_loader.SRC] + [os.path.join(CSRC, f) for f in ("tg_eval.h", "tg_sqp.h", "tg_spec.h", "tg_smooth.h")]
    if not os.path.exists(out) or any(os.path.getmtime(out) < os.path.getmtime(d) for d in deps):
        subprocess.run(["g++", "-std=c++14", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-Wno-unknown-pragmas",
                        "-DTG_WITH_SQP"] + list(flags) + ["-o", out, SRC], check=True, capture_output=True)
    return HostSimKKT(out)


def scipy_core_multipliers(hs, pp, maxiter=100, acc=1e-6):
    """hostsim_loader.scipy_core_solve's loop (scipy/optimize/_slsqp_py.py:524-555, analytic host-sim evaluations),
    returning dict(x, status, nit, multipliers = mult[:m]): OptimizeResult.multipliers of the last QP."""
    from scipy.optimize._slsqplib import slsqp
    L = pp.layout
    n, m, meq = L.n, L.m, L.meq
    x = np.clip(pp.x0, pp.xl, pp.xu).copy()
    xl = pp.xl.copy(); xu = pp.xu.copy()
    xl[~np.isfinite(xl)] = np.nan; xu[~np.isfinite(xu)] = np.nan
    state = {"acc": acc, "alpha": 0.0, "f0": 0.0, "gs": 0.0, "h1": 0.0, "h2": 0.0, "h3": 0.0, "h4": 0.0, "t": 0.0,
             "t0": 0.0, "tol": 10.0 * acc, "exact": 0, "inconsistent": 0, "reset": 0, "iter": 0,
             "itermax": int(maxiter), "line": 0, "m": m, "meq": meq, "mode": 0, "n": n}
    indices = np.zeros(max(m + 2 * n + 2, 1), dtype=np.int32)
    size = n * (n + 1) // 2 + 3 * m * n - (m + 5 * n + 7) * meq + 9 * m + 8 * n * n + 35 * n + meq * meq + 28
    if m - meq == 0:
        size += 2 * n * (n + 1)
    buffer = np.zeros(max(size, 1)); mult = np.zeros(max(1, m + 2 * n + 2))
    C = np.zeros((max(1, m), n), order="F"); d = np.zeros(max(1, m))
    fx, g, c, J = hs.eval(pp, x)
    C[:m, :] = J; d[:m] = c; g = g.copy()
    while True:
        slsqp(state, fx, g, C, d, x, mult, xl, xu, buffer, indices)
        if state["mode"] == 1:
            fx, _, c, _ = hs.eval(pp, x, jac=False)
            d[:m] = c
        if state["mode"] == -1:
            _, g, _, J = hs.eval(pp, x)
            g = g.copy(); C[:m, :] = J
        if abs(state["mode"]) != 1:
            break
    return dict(x=x, status=int(state["mode"]), nit=int(state["iter"]), multipliers=mult[:m].copy())
