"""TEST INFRASTRUCTURE: the host build of tests/hostsim/tg_hostsim_polish.cpp (tg_hostsim_kkt.cpp plus the post-solve
polish of csrc/tg_polish.h).  The product never loads it."""
import ctypes
import os
import subprocess

import numpy as np

import hostsim_kkt
import hostsim_loader
from hostsim_loader import ND, NI, CSRC, HERE

SRC = os.path.join(HERE, "hostsim", "tg_hostsim_polish.cpp")


class HostSimPolish(hostsim_kkt.HostSimKKT):
    def polish(self, pp, sol, maxiter=8, tol=1e-8):
        """tg_polish_problem on a copy of sol (a solve_kkt result): dict(x, f, violation, lam, kkt, polish_status,
        polish_iters)"""
        L = pp.layout
        x = np.array(sol["x"], dtype=np.float64); f = np.array([sol["f"]], dtype=np.float64)
        viol = np.array([sol.get("violation", 0)], dtype=np.int32)
        lam = np.zeros(max(L.m, 1)); lam[:L.m] = sol["lam"]
        kkt = np.array(sol["kkt"], dtype=np.float64)
        ps = np.zeros(1, np.int32); pi = np.zeros(1, np.int32)
        self.lib.hs_polish.argtypes = [NI, ND, ND, ND, ctypes.c_int, NI, ND, ND, NI, NI, ctypes.c_int, ctypes.c_double]
        self.lib.hs_polish(pp.spec, pp.par, x, f, int(sol["status"]), viol, lam, kkt, ps, pi, int(maxiter), float(tol))
        return dict(x=x, f=f[0], violation=int(viol[0]), lam=lam[:L.m], kkt=kkt, polish_status=int(ps[0]),
                    polish_iters=int(pi[0]))


def load():
    out = os.path.join(HERE, "hostsim", "_build_hostsim_polish.so")
    deps = [SRC, hostsim_kkt.SRC, hostsim_loader.SRC] + [os.path.join(CSRC, f) for f in (
        "tg_eval.h", "tg_sqp.h", "tg_spec.h", "tg_smooth.h", "tg_polish.h")]
    if not os.path.exists(out) or any(os.path.getmtime(out) < os.path.getmtime(d) for d in deps):
        subprocess.run(["g++", "-std=c++14", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-Wno-unknown-pragmas",
                        "-DTG_WITH_SQP", "-o", out, SRC], check=True, capture_output=True)
    return HostSimPolish(out)
