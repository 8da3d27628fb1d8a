"""Batched entry points over the CUDA library: device-resident (torch tensors as buffers) and
host-buffer (numpy, copies inside the C call) variants of

  * ``evaluate``  -- M1: objective, gradient, SLSQP-ordered constraint rows and analytic Jacobian
    rows of the nonlinear constraints, for B problems of one shape; what the reference computes with
    1 + (n+1) Python calls of every closure per SLSQP iteration (TG/trajectory_generator.py:171-250
    under scipy's finite differences);
  * ``solve``     -- M2: the scipy SLSQP call of TG/trajectory_generator.py:87-94 for B problems.

PyTorch is used only to own device memory and streams.
"""
import ctypes

import numpy as np

from . import _native
from .problem import Layout

JACOBIAN_MODES = {"analytic": 0, "fd": 1}     # "fd": scipy's forward differences emulated on the GPU


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


def solve(spec, par, x, maxiter=100, ftol=1e-6, jacobian="analytic", buffers=None, fused=False):
    """Device-resident M2 solve.  x [B,n] is overwritten with the optimised variables.
    Returns dict(x, f, status, nit, violation) of CUDA tensors.
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
    with torch.cuda.device(dev):
        rc = _native.lib().tg_solve_batch(buf.sp, B, _ptr(par), _ptr(x), _ptr(buf.f), _ptr(buf.status), _ptr(buf.nit),
                                          _ptr(buf.violation), int(maxiter), float(ftol), _flags(jacobian, fused),
                                          _ptr(buf.ws), buf.ws.numel(), _stream(torch, dev))
    _native.check(rc, "tg_solve_batch")
    return dict(x=x, f=buf.f, status=buf.status, nit=buf.nit, violation=buf.violation)


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


def solve_mixed(buckets, maxiter=100, ftol=1e-6, jacobian="analytic"):
    """Device-resident M2 solve of problems of DIFFERENT shapes in one call (tg_solve_mixed_batch).
    buckets: list of (spec, par [Bk, P], x [Bk, n]) CUDA tensors; x is overwritten with the solution.  The buckets run
    concurrently on internal streams that fork from and join the current stream.  Returns one dict(x, f, status, nit,
    violation) of CUDA tensors per bucket."""
    torch = _torch()
    L = _native.lib()
    nb = len(buckets)
    if nb == 0:
        return []
    nspec = L.tg_spec_count()
    specs = np.zeros((nb, nspec), dtype=np.int32)
    counts = np.zeros(nb, dtype=np.int32)
    vp_array = ctypes.c_void_p * nb
    ptrs = {k: vp_array() for k in ("par", "x", "f", "status", "nit", "violation")}
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
        outs.append(out); keep.append(par)
        ptrs["par"][k] = par.data_ptr()
        for name in ("x", "f", "status", "nit", "violation"):
            ptrs[name][k] = out[name].data_ptr()
    L.tg_solve_mixed_batch.restype = ctypes.c_int
    L.tg_solve_mixed_batch.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p] + [ctypes.c_void_p] * 6 + \
                                      [ctypes.c_int, ctypes.c_double, ctypes.c_int, ctypes.c_void_p]
    with torch.cuda.device(dev):
        rc = L.tg_solve_mixed_batch(nb, specs.ctypes.data, counts.ctypes.data, ptrs["par"], ptrs["x"], ptrs["f"], ptrs["status"],
                                    ptrs["nit"], ptrs["violation"], int(maxiter), float(ftol), _flags(jacobian, False),
                                    _stream(torch, dev))
    _native.check(rc, "tg_solve_mixed_batch")
    return outs
