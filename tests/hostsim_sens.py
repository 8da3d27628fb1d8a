"""TEST INFRASTRUCTURE: the host build of tests/hostsim/tg_hostsim_sens.cpp (tg_hostsim_polish.cpp plus the parameter
sensitivities of csrc/tg_sens.h).  The product never loads it."""
import ctypes
import os
import subprocess

import numpy as np

import hostsim_kkt
import hostsim_loader
import hostsim_polish
from hostsim_loader import ND, NI, CSRC, HERE

SRC = os.path.join(HERE, "hostsim", "tg_hostsim_sens.cpp")


class HostSimSens(hostsim_polish.HostSimPolish):
    def sensitivity(self, pp, sol, x_bar, f_bar=0.0, tol=1e-6):
        """tg_sens_problem on sol (a solve_kkt or polish result): (par_bar [P], sens_status)"""
        L = pp.layout
        lam = np.zeros(max(L.m, 1)); lam[:L.m] = sol["lam"]
        pbar = np.zeros(max(L.P, 1)); st = np.zeros(1, np.int32)
        self.lib.hs_sens.argtypes = [NI, ND, ND, ctypes.c_int, ND, ND, ctypes.c_double, ND, NI, ctypes.c_double]
        self.lib.hs_sens(pp.spec, np.ascontiguousarray(pp.par, dtype=np.float64),
                         np.ascontiguousarray(sol["x"], dtype=np.float64), int(sol["status"]), lam,
                         np.ascontiguousarray(x_bar, dtype=np.float64), float(f_bar), pbar, st, float(tol))
        return pbar[:L.P], int(st[0])


def load():
    out = os.path.join(HERE, "hostsim", "_build_hostsim_sens.so")
    deps = [SRC, hostsim_polish.SRC, hostsim_kkt.SRC, hostsim_loader.SRC] + [os.path.join(CSRC, f) for f in (
        "tg_eval.h", "tg_sqp.h", "tg_spec.h", "tg_smooth.h", "tg_polish.h", "tg_sens.h")]
    if not os.path.exists(out) or any(os.path.getmtime(out) < os.path.getmtime(d) for d in deps):
        subprocess.run(["g++", "-std=c++14", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-Wno-unknown-pragmas",
                        "-DTG_WITH_SQP", "-o", out, SRC], check=True, capture_output=True)
    return HostSimSens(out)
