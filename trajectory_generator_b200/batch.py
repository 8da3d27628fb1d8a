"""Batched entry points over the CUDA library: device-resident (torch tensors as buffers) and
host-buffer (numpy, copies inside the C call) variants of

  * ``evaluate``  -- M1: objective, gradient, SLSQP-ordered constraint rows and analytic Jacobian
    rows of the nonlinear constraints, for B problems of one shape; what the reference computes with
    1 + (n+1) Python calls of every closure per SLSQP iteration (TG/trajectory_generator.py:171-250
    under scipy's finite differences);
  * ``solve``     -- M2: the scipy SLSQP call of TG/trajectory_generator.py:87-94 for B problems;
  * ``solve_multistart`` -- M2 from K seeded starts per problem, the best converged feasible result kept (opt-in).

Every solve entry point takes ``multipliers=False``; with True its result also holds ``lam`` [B, m], the KKT
multipliers of the last QP in constraint row order (scipy's ``OptimizeResult.multipliers``; ``Layout.row_blocks`` names
the rows), and ``kkt`` [B, 4], the first-order optimality certificate at the returned x (KKT_FIELDS; DESIGN.md §4).

PyTorch is used only to own device memory and streams.
"""
import ctypes

import numpy as np

from . import _native
from .problem import Layout

JACOBIAN_MODES = {"analytic": 0, "fd": 1}     # "fd": scipy's forward differences emulated on the GPU
# entries of `kkt` (include/trajectory_generator_b200.h, tg_solve_batch_kkt): absolute, NaN = +inf
KKT_FIELDS = ("stationarity", "infeasibility", "dual_infeasibility", "complementarity")


def _torch():
    import torch
    return torch


def _ptr(t):
    return ctypes.c_void_p(0 if t is None else t.data_ptr())


def _stream(torch, device):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def evaluate(spec, par, x, want=("f", "g", "c", "jnl"), out=None):
    """Device-resident M1 evaluation.  par [B,P], x [B,n]: float64 CUDA tensors.  Returns a dict of CUDA tensors."""
    torch = _torch()
    lay = Layout(spec)
    if not (par.is_cuda and x.is_cuda):
        raise RuntimeError("evaluate() needs CUDA tensors (there is no CPU path); use evaluate_host for numpy input")
    B = x.shape[0]
    par = par.contiguous(); x = x.contiguous()
    assert par.dtype == torch.float64 and x.dtype == torch.float64
    assert par.shape == (B, lay.P) and x.shape == (B, lay.n)
    dev = x.device
    res = out if out is not None else {}
    shapes = {"f": (B,), "g": (B, lay.n), "c": (B, lay.m), "jnl": (B, lay.m_nl, lay.n)}
    for k in want:
        if k not in res:
            res[k] = torch.empty(shapes[k], dtype=torch.float64, device=dev)
    spec, sp = _native.spec_ptr(spec)
    with torch.cuda.device(dev):
        rc = _native.lib().tg_eval_batch(sp, B, _ptr(par), _ptr(x), _ptr(res.get("f")), _ptr(res.get("g")),
                                         _ptr(res.get("c")), _ptr(res.get("jnl")), _stream(torch, dev))
    _native.check(rc, "tg_eval_batch")
    return res


def linear_rows(spec, par):
    """Constant Jacobian rows of the linear blocks: [B, m, n] CUDA tensor (nonlinear rows are zero)."""
    torch = _torch()
    lay = Layout(spec)
    B = par.shape[0]
    par = par.contiguous()
    A = torch.zeros((B, lay.m, lay.n), dtype=torch.float64, device=par.device)
    spec, sp = _native.spec_ptr(spec)
    with torch.cuda.device(par.device):
        rc = _native.lib().tg_linear_rows_batch(sp, B, _ptr(par), _ptr(A), _stream(torch, par.device))
    _native.check(rc, "tg_linear_rows_batch")
    return A


class SolveBuffers:
    """Reusable device buffers of one solve shape (outputs + the kernel's scratch)."""

    def __init__(self, spec, B, device):
        torch = _torch()
        self.spec, self.sp = _native.spec_ptr(spec)
        self.B = B
        self.f = torch.empty(B, dtype=torch.float64, device=device)
        self.status = torch.empty(B, dtype=torch.int32, device=device)
        self.nit = torch.empty(B, dtype=torch.int32, device=device)
        self.violation = torch.empty(B, dtype=torch.int32, device=device)
        with torch.cuda.device(device):
            nbytes = _native.lib().tg_solve_workspace_bytes(self.sp, B)
        if nbytes == 0:
            raise RuntimeError("tg_solve_workspace_bytes: %s" % _native.lib().tg_last_error().decode())
        self.ws = torch.empty(nbytes, dtype=torch.uint8, device=device)


PLAN_FIELDS = ("gs_ls", "gs_qp", "staged", "qp_far", "ls_far", "slots", "slot_kib")


def solve_plan(spec, B):
    """Launch plan of the lock-step solve of B problems of this shape on the current device (tg_solve_plan_info): lanes
    per problem of the line-search and QP stages, whether the QP stage stages the state in shared memory, whether the
    QP / line-search scratch lives in workspace slots (shapes whose scratch does not fit in shared memory), the number
    of slots and their KiB.  A dict keyed by PLAN_FIELDS."""
    spec, sp = _native.spec_ptr(spec)
    out = np.zeros(len(PLAN_FIELDS), dtype=np.int32)
    cnt = _native.lib().tg_solve_plan_info(sp, int(B), out.ctypes.data_as(_native._I32), out.size)
    _native.check(-cnt if cnt < 0 else 0, "tg_solve_plan_info")
    return {k: int(v) for k, v in zip(PLAN_FIELDS, out)}


def _flags(jacobian, fused):
    return JACOBIAN_MODES[jacobian] | (2 if fused else 0)


def _kkt_outputs(torch, lay, B, dev):
    return dict(lam=torch.empty((B, lay.m), dtype=torch.float64, device=dev),
                kkt=torch.empty((B, 4), dtype=torch.float64, device=dev))


def solve(spec, par, x, maxiter=100, ftol=1e-6, jacobian="analytic", buffers=None, fused=False, multipliers=False):
    """Device-resident M2 solve.  x [B,n] is overwritten with the optimised variables.
    Returns dict(x, f, status, nit, violation) of CUDA tensors; with multipliers=True also lam [B, m] and kkt [B, 4]
    (tg_solve_batch_kkt), new tensors of every call.
    fused=False (default): lock-step stage kernels over the whole batch; fused=True: one persistent kernel in
    which each warp runs a whole solve (same arithmetic, kept for comparison)."""
    torch = _torch()
    lay = Layout(spec)
    if not (par.is_cuda and x.is_cuda):
        raise RuntimeError("solve() needs CUDA tensors (there is no CPU path); use solve_host for numpy input")
    B = x.shape[0]
    if par.dtype != torch.float64 or x.dtype != torch.float64:
        raise ValueError("solve() needs float64 tensors, got %s / %s" % (par.dtype, x.dtype))
    if par.device != x.device:
        raise ValueError("par and x live on different devices")
    if not (par.is_contiguous() and x.is_contiguous()) or par.shape != (B, lay.P) or x.shape != (B, lay.n):
        raise ValueError("par [B, %d] and x [B, %d] must be contiguous tensors of the descriptor's shape" % (lay.P, lay.n))
    dev = x.device
    buf = buffers if buffers is not None else SolveBuffers(spec, B, dev)
    if buf.B < B or not np.array_equal(buf.spec, np.ascontiguousarray(spec, dtype=np.int32)) or buf.ws.device != dev:
        raise ValueError("the SolveBuffers were made for another shape, a smaller batch or another device")
    args = (buf.sp, B, _ptr(par), _ptr(x), _ptr(buf.f), _ptr(buf.status), _ptr(buf.nit), _ptr(buf.violation),
            int(maxiter), float(ftol), _flags(jacobian, fused), _ptr(buf.ws), buf.ws.numel(), _stream(torch, dev))
    extra = _kkt_outputs(torch, lay, B, dev) if multipliers else {}
    with torch.cuda.device(dev):
        if multipliers:
            rc = _native.lib().tg_solve_batch_kkt(*args, _ptr(extra["lam"]), _ptr(extra["kkt"]))
        else:
            rc = _native.lib().tg_solve_batch(*args)
    _native.check(rc, "tg_solve_batch_kkt" if multipliers else "tg_solve_batch")
    return dict(x=x, f=buf.f, status=buf.status, nit=buf.nit, violation=buf.violation, **extra)


def _np_ptr(a):
    return ctypes.c_void_p(0 if a is None else a.ctypes.data)


def pinned_empty(shape, dtype=np.float64):
    """numpy array backed by page-locked host memory (torch owns it): the host-buffer entry points copy such buffers with
    the DMA engines asynchronously and pipeline a batch in chunks; pageable arrays work too, one synchronous chunk."""
    torch = _torch()
    t = torch.empty(tuple(shape), dtype={np.float64: torch.float64, np.int32: torch.int32}[dtype]).pin_memory()
    return t.numpy()


def evaluate_host(spec, par, x, want=("f", "g", "c", "jnl"), out=None):
    """Host-buffer M1 evaluation through tg_eval_host (numpy in, numpy out; copies inside the call).  `out`: dict of
    arrays to write into (e.g. ``pinned_empty`` buffers kept between calls); missing entries are allocated."""
    lay = Layout(spec)
    par = np.ascontiguousarray(par, dtype=np.float64).reshape(-1, lay.P)
    x = np.ascontiguousarray(x, dtype=np.float64).reshape(-1, lay.n)
    B = x.shape[0]
    shapes = {"f": (B,), "g": (B, lay.n), "c": (B, lay.m), "jnl": (B, lay.m_nl, lay.n)}
    res = out if out is not None else {}
    for k in want:
        if k not in res:
            res[k] = np.empty(shapes[k])
        elif res[k].shape != shapes[k] or res[k].dtype != np.float64 or not res[k].flags.c_contiguous:
            raise ValueError("out[%r] must be a contiguous float64 array of shape %r" % (k, shapes[k]))
    spec, sp = _native.spec_ptr(spec)
    rc = _native.lib().tg_eval_host(sp, B, _np_ptr(par), _np_ptr(x), _np_ptr(res.get("f")), _np_ptr(res.get("g")),
                                    _np_ptr(res.get("c")), _np_ptr(res.get("jnl")))
    _native.check(rc, "tg_eval_host")
    return res


def solve_host(spec, par, x0, maxiter=100, ftol=1e-6, jacobian="analytic", fused=False):
    """Host-buffer M2 solve through tg_solve_host.  Returns dict(x, f, status, nit, violation) of numpy arrays."""
    lay = Layout(spec)
    par = np.ascontiguousarray(par, dtype=np.float64).reshape(-1, lay.P)
    x = np.array(x0, dtype=np.float64).reshape(-1, lay.n)
    B = x.shape[0]
    f = np.empty(B); status = np.empty(B, dtype=np.int32); nit = np.empty(B, dtype=np.int32)
    viol = np.empty(B, dtype=np.int32)
    spec, sp = _native.spec_ptr(spec)
    rc = _native.lib().tg_solve_host(sp, B, _np_ptr(par), _np_ptr(x), _np_ptr(f), _np_ptr(status), _np_ptr(nit),
                                     _np_ptr(viol), int(maxiter), float(ftol), _flags(jacobian, fused))
    _native.check(rc, "tg_solve_host")
    return dict(x=x, f=f, status=status, nit=nit, violation=viol)


def solve_mixed_host(buckets, maxiter=100, ftol=1e-6, jacobian="analytic"):
    """Host-buffer M2 solve of problems of DIFFERENT shapes in one call (tg_solve_mixed_host, SURVEY.md 8(f) f3).
    buckets: list of (spec, par[Bk,P], x0[Bk,n]).  Buckets run concurrently on the device, each on its own stream.
    Returns one dict(x, f, status, nit, violation) of numpy arrays per bucket, in input order."""
    L = _native.lib()
    nb = len(buckets)
    if nb == 0:
        return []
    nspec = L.tg_spec_count()
    specs = np.zeros((nb, nspec), dtype=np.int32)
    counts = np.zeros(nb, dtype=np.int32)
    keep, outs = [], []
    vp_array = ctypes.c_void_p * nb
    ptrs = {k: vp_array() for k in ("par", "x", "f", "status", "nit", "violation")}
    for k, (spec, par, x0) in enumerate(buckets):
        lay = Layout(spec)
        spec = np.ascontiguousarray(spec, dtype=np.int32)
        if spec.size != nspec:
            raise ValueError("spec must have %d entries" % nspec)
        specs[k] = spec
        par = np.ascontiguousarray(par, dtype=np.float64).reshape(-1, lay.P)
        x = np.array(x0, dtype=np.float64).reshape(-1, lay.n)
        B = x.shape[0]
        if par.shape[0] != B:
            raise ValueError("bucket %d: %d parameter rows for %d problems" % (k, par.shape[0], B))
        counts[k] = B
        out = dict(x=x, f=np.empty(B), status=np.empty(B, dtype=np.int32), nit=np.empty(B, dtype=np.int32),
                   violation=np.empty(B, dtype=np.int32))
        keep.append(par)
        outs.append(out)
        ptrs["par"][k] = par.ctypes.data
        for name in ("x", "f", "status", "nit", "violation"):
            ptrs[name][k] = out[name].ctypes.data
    L.tg_solve_mixed_host.restype = ctypes.c_int
    L.tg_solve_mixed_host.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p] + [ctypes.c_void_p] * 6 + \
                                     [ctypes.c_int, ctypes.c_double, ctypes.c_int]
    rc = L.tg_solve_mixed_host(nb, specs.ctypes.data, counts.ctypes.data, ptrs["par"], ptrs["x"], ptrs["f"], ptrs["status"],
                               ptrs["nit"], ptrs["violation"], int(maxiter), float(ftol), _flags(jacobian, False))
    _native.check(rc, "tg_solve_mixed_host")
    return outs


def solve_mixed(buckets, maxiter=100, ftol=1e-6, jacobian="analytic", multipliers=False):
    """Device-resident M2 solve of problems of DIFFERENT shapes in one call (tg_solve_mixed_batch).
    buckets: list of (spec, par [Bk, P], x [Bk, n]) CUDA tensors; x is overwritten with the solution.  The buckets run
    concurrently on internal streams that fork from and join the current stream.  Returns one dict(x, f, status, nit,
    violation) of CUDA tensors per bucket; with multipliers=True each also holds lam [Bk, m] and kkt [Bk, 4]
    (tg_solve_mixed_batch_kkt)."""
    torch = _torch()
    L = _native.lib()
    nb = len(buckets)
    if nb == 0:
        return []
    nspec = L.tg_spec_count()
    specs = np.zeros((nb, nspec), dtype=np.int32)
    counts = np.zeros(nb, dtype=np.int32)
    vp_array = ctypes.c_void_p * nb
    ptrs = {k: vp_array() for k in ("par", "x", "f", "status", "nit", "violation", "lam", "kkt")}
    outs, keep = [], []
    dev = buckets[0][2].device
    for k, (spec, par, x) in enumerate(buckets):
        lay = Layout(spec)
        if not (par.is_cuda and x.is_cuda) or par.device != dev or x.device != dev:
            raise RuntimeError("solve_mixed() needs CUDA tensors on one device (there is no CPU path)")
        if par.dtype != torch.float64 or x.dtype != torch.float64:
            raise ValueError("solve_mixed() needs float64 tensors")
        B = x.shape[0]
        if not (par.is_contiguous() and x.is_contiguous()) or par.shape != (B, lay.P) or x.shape != (B, lay.n):
            raise ValueError("bucket %d: par / x do not have the shapes of the descriptor" % k)
        specs[k] = np.ascontiguousarray(spec, dtype=np.int32)
        counts[k] = B
        out = dict(x=x, f=torch.empty(B, dtype=torch.float64, device=dev), status=torch.empty(B, dtype=torch.int32, device=dev),
                   nit=torch.empty(B, dtype=torch.int32, device=dev), violation=torch.empty(B, dtype=torch.int32, device=dev))
        if multipliers:
            out.update(_kkt_outputs(torch, lay, B, dev))
        outs.append(out); keep.append(par)
        ptrs["par"][k] = par.data_ptr()
        for name in ("x", "f", "status", "nit", "violation") + (("lam", "kkt") if multipliers else ()):
            ptrs[name][k] = out[name].data_ptr()
    args = (nb, specs.ctypes.data, counts.ctypes.data, ptrs["par"], ptrs["x"], ptrs["f"], ptrs["status"], ptrs["nit"],
            ptrs["violation"], int(maxiter), float(ftol), _flags(jacobian, False), _stream(torch, dev))
    name = "tg_solve_mixed_batch_kkt" if multipliers else "tg_solve_mixed_batch"
    fn = getattr(L, name)
    fn.restype = ctypes.c_int
    fn.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p] + [ctypes.c_void_p] * 6 + \
        [ctypes.c_int, ctypes.c_double, ctypes.c_int, ctypes.c_void_p] + [ctypes.c_void_p] * (2 if multipliers else 0)
    with torch.cuda.device(dev):
        rc = fn(*args, ptrs["lam"], ptrs["kkt"]) if multipliers else fn(*args)
    _native.check(rc, name)
    return outs


# ---------------------------------------------------------------------------------------------------------------------
# Multi-start solves (include/trajectory_generator_b200.h, DESIGN.md §4 *Multi-start*): K seeded starts per problem are
# solved as ordinary problems and the best converged feasible one is kept.
# ---------------------------------------------------------------------------------------------------------------------
MULTISTART_SPREAD = 0.25    # offset scale of the interior control points, relative to |P_{N-1} - P_0| (DESIGN.md §4)
MULTISTART_TOL = 1e-5       # feasibility tolerance of the selection: the reference's is_violation tolerance (10e-6)
MULTISTART_ROWS = 1 << 20   # cap of the B * K rows expanded at a time (par is replicated: B * K * P doubles)


def _check_device_rows(what, spec, par, x, starts=1):
    """(layout, B) of par [B, P] and x [B * starts, n]: contiguous float64 CUDA tensors on one device"""
    torch = _torch()
    lay = Layout(spec)
    if not (par.is_cuda and x.is_cuda):
        raise RuntimeError("%s needs CUDA tensors (there is no CPU path)" % what)
    if par.dtype != torch.float64 or x.dtype != torch.float64:
        raise ValueError("%s needs float64 tensors, got %s / %s" % (what, par.dtype, x.dtype))
    if par.device != x.device:
        raise ValueError("par and x live on different devices")
    B = par.shape[0]
    if not (par.is_contiguous() and x.is_contiguous()) or par.shape != (B, lay.P) or x.shape != (B * starts, lay.n):
        raise ValueError("par [B, %d] and x [B * %d, %d] must be contiguous tensors of the descriptor's shape"
                         % (lay.P, starts, lay.n))
    return lay, B


def multistart_expand(spec, par, x0, starts, seed=0, spread=MULTISTART_SPREAD):
    """Starts of B problems (tg_multistart_expand): par [B, P], x0 [B, n] float64 CUDA tensors ->
    (par_out [B*K, P], x_out [B*K, n]); row b*K + k is start k of problem b, start 0 is x0[b] bit for bit."""
    torch = _torch()
    lay, B = _check_device_rows("multistart_expand()", spec, par, x0)
    K = int(starts)
    if K < 1:
        raise ValueError("starts must be at least 1")
    dev = x0.device
    par_out = torch.empty((B * K, lay.P), dtype=torch.float64, device=dev)
    x_out = torch.empty((B * K, lay.n), dtype=torch.float64, device=dev)
    spec, sp = _native.spec_ptr(spec)
    with torch.cuda.device(dev):
        rc = _native.lib().tg_multistart_expand(sp, B, K, _ptr(par), _ptr(x0), int(seed) & (2 ** 64 - 1), float(spread),
                                                _ptr(par_out), _ptr(x_out), _stream(torch, dev))
    _native.check(rc, "tg_multistart_expand")
    return par_out, x_out


def multistart_select(spec, par, sol, starts, tol=MULTISTART_TOL, out=None):
    """Best start per problem (tg_multistart_select).  par [B, P]: the problems' rows; sol: the dict a solve of the
    B*K expanded rows returned.  Returns dict(x, f, status, nit, violation, best_start, max_violation) with B rows and
    `start_max_violation` [B, K] (the true maximum violation of every start); `out` may hold any of these to write into."""
    torch = _torch()
    K = int(starts)
    if K < 1:
        raise ValueError("starts must be at least 1")
    lay, B = _check_device_rows("multistart_select()", spec, par, sol["x"], K)
    dev = par.device
    res = {} if out is None else out
    shapes = dict(x=((B, lay.n), torch.float64), f=((B,), torch.float64), status=((B,), torch.int32),
                  nit=((B,), torch.int32), violation=((B,), torch.int32), best_start=((B,), torch.int32),
                  start_max_violation=((B, K), torch.float64))
    for k, (shape, dtype) in shapes.items():
        if k not in res:
            res[k] = torch.empty(shape, dtype=dtype, device=dev)
    spec, sp = _native.spec_ptr(spec)
    with torch.cuda.device(dev):
        rc = _native.lib().tg_multistart_select(
            sp, B, K, _ptr(par), _ptr(sol["x"]), _ptr(sol["f"]), _ptr(sol["status"]), _ptr(sol["nit"]),
            _ptr(sol["violation"]), float(tol), _ptr(res["x"]), _ptr(res["f"]), _ptr(res["status"]), _ptr(res["nit"]),
            _ptr(res["violation"]), _ptr(res["best_start"]), _ptr(res["start_max_violation"]), _stream(torch, dev))
    _native.check(rc, "tg_multistart_select")
    res["max_violation"] = res["start_max_violation"].gather(1, res["best_start"].long()[:, None])[:, 0]
    return res


def solve_mixed_multistart(buckets, starts, seed=0, spread=MULTISTART_SPREAD, tol=MULTISTART_TOL, maxiter=100,
                           ftol=1e-6, jacobian="analytic", return_all=False, multipliers=False):
    """Multi-start solve of problems of one or several shapes: buckets = list of (spec, par [Bk, P], x0 [Bk, n]) CUDA
    tensors (x0 is not modified).  Per bucket: expand -> solve -> select on the current stream, in pieces of at most
    MULTISTART_ROWS expanded rows; the pieces of several shapes go through one ``solve_mixed`` call.  Returns one dict
    per bucket: the B-row dict of ``solve`` plus best_start and max_violation (the winner's true maximum violation);
    with return_all, also "all": the K per-start results, dict(x [B, K, n], f, status, nit, violation,
    max_violation [B, K]).  multipliers=True adds the winner's lam [B, m] and kkt [B, 4] (and every start's,
    [B, K, m] and [B, K, 4], under "all")."""
    torch = _torch()
    K = int(starts)
    if K < 1:
        raise ValueError("starts must be at least 1")
    outs, pieces = [], []
    for j, (spec, par, x0) in enumerate(buckets):
        lay, B = _check_device_rows("solve_multistart()", spec, par, x0)
        dev = x0.device
        res = dict(x=torch.empty_like(x0), f=torch.empty(B, dtype=torch.float64, device=dev))
        for k in ("status", "nit", "violation", "best_start"):
            res[k] = torch.empty(B, dtype=torch.int32, device=dev)
        res["start_max_violation"] = torch.empty((B, K), dtype=torch.float64, device=dev)
        if multipliers:
            res.update(_kkt_outputs(torch, lay, B, dev))
        if return_all:
            res["all"] = dict(x=torch.empty((B, K, lay.n), dtype=torch.float64, device=dev),
                              f=torch.empty((B, K), dtype=torch.float64, device=dev),
                              **{k: torch.empty((B, K), dtype=torch.int32, device=dev) for k in ("status", "nit", "violation")})
            if multipliers:
                res["all"].update(lam=torch.empty((B, K, lay.m), dtype=torch.float64, device=dev),
                                  kkt=torch.empty((B, K, 4), dtype=torch.float64, device=dev))
        outs.append(res)
        per = max(1, MULTISTART_ROWS // K)
        pieces += [(j, lo, min(B, lo + per)) for lo in range(0, B, per)]
    waves, rows = [[]], 0
    for j, lo, hi in pieces:
        if waves[-1] and rows + (hi - lo) * K > MULTISTART_ROWS:
            waves.append([])
            rows = 0
        waves[-1].append((j, lo, hi))
        rows += (hi - lo) * K
    for wave in waves:
        if not wave:
            continue
        expanded = []
        for j, lo, hi in wave:
            spec, par, x0 = buckets[j]
            expanded.append((spec,) + multistart_expand(spec, par[lo:hi], x0[lo:hi], K, seed, spread))
        if len(expanded) == 1:
            sols = [solve(*expanded[0], maxiter=maxiter, ftol=ftol, jacobian=jacobian, multipliers=multipliers)]
        else:
            sols = solve_mixed(expanded, maxiter, ftol, jacobian, multipliers)
        for (j, lo, hi), sol in zip(wave, sols):
            spec, par, _ = buckets[j]
            res = outs[j]
            multistart_select(spec, par[lo:hi], sol, K, tol, out={k: res[k][lo:hi] for k in (
                "x", "f", "status", "nit", "violation", "best_start", "start_max_violation")})
            if multipliers:
                rows = torch.arange(hi - lo, device=par.device) * K + res["best_start"][lo:hi].long()
                res["lam"][lo:hi] = sol["lam"][rows]
                res["kkt"][lo:hi] = sol["kkt"][rows]
            if return_all:
                for k in ("x", "f", "status", "nit", "violation") + (("lam", "kkt") if multipliers else ()):
                    res["all"][k][lo:hi] = sol[k].view(res["all"][k][lo:hi].shape)
    for res in outs:
        mv = res.pop("start_max_violation")
        res["max_violation"] = mv.gather(1, res["best_start"].long()[:, None])[:, 0]
        if return_all:
            res["all"]["max_violation"] = mv
    return outs


def solve_multistart(spec, par, x0, starts, seed=0, spread=MULTISTART_SPREAD, tol=MULTISTART_TOL, maxiter=100, ftol=1e-6,
                     jacobian="analytic", return_all=False, multipliers=False):
    """Multi-start solve of B problems of one shape (see ``solve_mixed_multistart``).  starts = 1 returns exactly what
    ``solve`` returns for x0 (start 0 is x0 itself), plus best_start = 0 and max_violation."""
    return solve_mixed_multistart([(spec, par, x0)], starts, seed, spread, tol, maxiter, ftol, jacobian, return_all,
                                  multipliers)[0]
