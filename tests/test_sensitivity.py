"""Parameter sensitivities of converged solves (csrc/tg_sens.h, tg_sens_batch; batch.sensitivity,
batch.solve_differentiable and BatchedProblem.solve(differentiable=True); DESIGN.md §4 *Sensitivities*).

CPU: the host build against a dense numpy restatement (the full KKT matrix solved with numpy.linalg.solve), against
re-solved points at perturbed parameters, the envelope identity, the statuses, and the error paths without a device.
GPU: the device against the host build; bit-identity across batch position, placement, instantiation and multi-start;
re-solve checks on synthetic batches; the autograd function and the front end."""
import numpy as np
import pytest

import helpers
import hostsim_sens
import problems
from trajectory_generator_b200.problem import pack_problem

H_REL = 6.0554544523933395e-06          # cbrt(DBL_EPSILON), the step of the device's central differences
CODES = {"ok": 0, "nonstrict": 1, "inexact": 2, "degenerate": 3, "skipped": 4, "nonfinite": 5, "indefinite": 6}
COMPUTED = (0, 1, 2)


def _fixture(name):
    d, cc, kw = problems.ALL[name](helpers.product_namespace())
    return pack_problem(d, cc, kw.get("objective_function_type", "minimal_velocity_and_time_path"),
                        kw.get("num_intervals_free_space"))


class _P:
    pass


def _with_par(pp, par):
    q = _P()
    q.spec, q.par, q.layout, q.x0, q.xl, q.xu = pp.spec, np.ascontiguousarray(par, np.float64), pp.layout, pp.x0, pp.xl, pp.xu
    return q


def _synthetic(name, count):
    from trajectory_generator_b200 import synthetic as syn
    bt = syn.make(name, count)
    L = bt.layout
    for i in range(count):
        pp = _P()
        pp.spec, pp.par, pp.x0, pp.layout = bt.spec, bt.par[i].copy(), bt.x0[i].copy(), L
        pp.xl = np.full(L.n, -np.inf); pp.xu = np.full(L.n, np.inf)
        pp.xl[L.ia:L.it0] = 10e-8
        if L.it0 < L.n:
            pp.xl[L.it0:] = 0; pp.xu[L.it0:] = L.N - 3
        yield pp


@pytest.fixture(scope="module")
def hostsim():
    return hostsim_sens.load()


def _polished(hs, pp):
    """the host solve and polish of pp, or None when the polish does not reach stationarity"""
    sol = hs.solve_kkt(pp)
    if sol["status"] != 0:
        return None
    out = hs.polish(pp, dict(sol, violation=0))
    return dict(out, status=0) if out["polish_status"] == 0 else None


def _stationary_cases(hs):
    """intermediate_curvature and sfc3d_four (a corridor problem) after the host polish, and polished C3 and C4 rows"""
    cases = [(n, _fixture(n)) for n in ("intermediate_curvature", "sfc3d_four")]
    cases += [("%s/%d" % (n, i), pp) for n in ("C3", "C4") for i, pp in enumerate(_synthetic(n, 3))]
    out = []
    for name, pp in cases:
        sol = _polished(hs, pp)
        if sol is not None:
            out.append((name, pp, sol))
    return out


def _bounds(pp):
    return np.where(np.isfinite(pp.xl), pp.xl, -np.inf), np.where(np.isfinite(pp.xu), pp.xu, np.inf)


def _sets(pp, x, lam):
    L = pp.layout
    xl, xu = _bounds(pp)
    free = np.flatnonzero((x != xl) & (x != xu))
    W = np.flatnonzero((np.arange(L.m) < L.meq) | (lam > 0))
    return free, W


def _dpar(hs, pp, x):
    """(dc/dp [m, P], dJ/dp [m, n, P]) at x by numpy central differences with the device's steps"""
    L = pp.layout
    dc = np.zeros((L.m, L.P)); dJ = np.zeros((L.m, L.n, L.P))
    for k in range(L.P):
        pk = pp.par[k]
        h = H_REL * max(1.0, abs(pk))
        res = []
        for v in (pk + h, pk - h):
            par = pp.par.copy(); par[k] = v
            _, _, c, J = hs.eval(_with_par(pp, par), x)
            res.append((c, J))
        den = (pk + h) - (pk - h)
        dc[:, k] = (res[0][0] - res[1][0]) / den
        dJ[:, :, k] = (res[0][1] - res[1][1]) / den
    return dc, dJ


def _restated(hs, pp, sol, x_bar, f_bar):
    """par_bar from the full KKT matrix [H A_W'; A_W 0] and numpy.linalg.solve"""
    x = sol["x"]
    f, g, c, J = hs.eval(pp, x)
    free, W = _sets(pp, x, sol["lam"])
    xl, xu = _bounds(pp)
    A = J[np.ix_(W, free)]
    lw = np.linalg.lstsq(A.T, g[free], rcond=None)[0]
    lam = np.zeros(pp.layout.m); lam[W] = lw
    H = np.zeros((len(free), len(free)))
    for b, i in enumerate(free):
        h = H_REL * max(1.0, abs(x[i]))
        xp, xm = min(x[i] + h, xu[i]), max(x[i] - h, xl[i])
        cols = []
        for xv in (xp, xm):
            y = x.copy(); y[i] = xv
            _, gy, _, Jy = hs.eval(pp, y)
            cols.append((gy - Jy.T @ lam)[free])
        H[:, b] = (cols[0] - cols[1]) / (xp - xm)
    H = 0.5 * (H + H.T)
    nF, nW = len(free), len(W)
    K = np.zeros((nF + nW, nF + nW))
    K[:nF, :nF] = H; K[:nF, nF:] = A.T; K[nF:, :nF] = A
    gbar = x_bar + f_bar * g
    sol_uw = np.linalg.solve(K, np.concatenate([gbar[free], np.zeros(nW)]))
    u, w = sol_uw[:nF], sol_uw[nF:]
    dc, dJ = _dpar(hs, pp, x)
    # d(grad_x L)/dp restricted to F, contracted with u, and dc_W/dp
    dgl = -np.einsum("j,jap->ap", lw, dJ[np.ix_(W, free, np.arange(pp.layout.P))])
    return -(u @ dgl) - w @ dc[W], lw, dc[W]


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def test_host_build_follows_the_dense_kkt_restatement(native_lib, hostsim):
    cases = _stationary_cases(hostsim)
    assert len(cases) >= 5, [c[0] for c in cases]
    rng = np.random.default_rng(11)
    for name, pp, sol in cases:
        x_bar, f_bar = rng.standard_normal(pp.layout.n), float(rng.standard_normal())
        pbar, st = hostsim.sensitivity(pp, sol, x_bar, f_bar)
        assert st in COMPUTED, (name, st)
        ref, _, _ = _restated(hostsim, pp, sol, x_bar, f_bar)
        assert np.abs(pbar - ref).max() <= 1e-7 * np.abs(ref).max(), (name, np.abs(pbar - ref).max(), np.abs(ref).max())


def _resolve_check(hs, pp, sol, pbar, x_bar, f_bar, direction, h=1e-5):
    """x_bar . dx + f_bar df along `direction` from the host polish started at x* at par +- h direction (maxiter 20,
    tol 1e-12); None when a re-solve is not replaced or the working sets differ.  (The polish stops at once at a
    stationary start, feasible or not, and where no Jacobian row of W reads the perturbed entries x* stays stationary:
    the start's multipliers are scaled by 1 + 1e-6 -- same working set -- so that Newton steps restore feasibility.)"""
    outs = []
    for s in (1, -1):
        q = _with_par(pp, pp.par + s * h * direction)
        f, g, c, J = hs.eval(q, sol["x"])
        start = dict(sol, f=f, lam=sol["lam"] * (1 + 1e-6), violation=0)
        out = hs.polish(q, start, maxiter=20, tol=1e-12)
        if out["polish_status"] not in (0, 1):
            return None
        outs.append(out)
    if not np.array_equal(_sets(pp, outs[0]["x"], outs[0]["lam"])[1], _sets(pp, sol["x"], sol["lam"])[1]) or \
            not np.array_equal(_sets(pp, outs[1]["x"], outs[1]["lam"])[1], _sets(pp, sol["x"], sol["lam"])[1]):
        return None
    fd = (x_bar @ (outs[0]["x"] - outs[1]["x"]) + f_bar * (outs[0]["f"] - outs[1]["f"])) / (2 * h)
    return fd, pbar @ direction


def test_host_build_against_re_solved_points(native_lib, hostsim):
    """the directional derivative against two polishes at perturbed parameters; sfc3d_four's corridor rows carry their
    parameters in their x-coefficients, so a psi without the linear rows' Jacobian fails here"""
    rng = np.random.default_rng(5)
    compared = set()
    for name, pp, sol in _stationary_cases(hostsim):
        x_bar, f_bar = rng.standard_normal(pp.layout.n), float(rng.standard_normal())
        pbar, st = hostsim.sensitivity(pp, sol, x_bar, f_bar)
        for trial in range(2):
            direction = rng.standard_normal(pp.layout.P) * np.maximum(1.0, np.abs(pp.par))
            r = _resolve_check(hostsim, pp, sol, pbar, x_bar, f_bar, direction)
            if r is None:
                continue
            fd, an = r
            assert abs(fd - an) <= 1e-4 * max(abs(fd), abs(an), 1e-3 * np.abs(pbar).max()), (name, fd, an)
            compared.add(name)
    assert "sfc3d_four" in compared and "intermediate_curvature" in compared, compared
    assert len(compared) >= 4, compared


def test_corridor_parameters_reach_par_bar(native_lib, hostsim):
    """the corridor block (rotation and bounds of the boxes) gets a nonzero gradient on sfc3d_four"""
    pp = _fixture("sfc3d_four")
    sol = _polished(hostsim, pp)
    L = pp.layout
    pbar, st = hostsim.sensitivity(pp, sol, np.ones(L.n), 1.0)
    assert st in COMPUTED
    assert np.abs(pbar[L.p_sfc:L.p_obs_c]).max() > 0


def test_envelope_identity_and_zero_upstream(native_lib, hostsim):
    for name, pp, sol in _stationary_cases(hostsim):
        zeros = np.zeros(pp.layout.n)
        pbar, st = hostsim.sensitivity(pp, sol, zeros, 1.0)
        assert st in COMPUTED
        _, lw, dcw = _restated(hostsim, pp, sol, zeros, 1.0)
        env = -lw @ dcw
        assert np.abs(pbar - env).max() <= 1e-8 * max(1.0, np.abs(env).max()), (name, np.abs(pbar - env).max())
        pz, st = hostsim.sensitivity(pp, sol, zeros, 0.0)
        assert st in COMPUTED and (pz == 0).all(), name


def test_statuses(native_lib, hostsim):
    # a row stopped by the iteration limit is skipped with a zero row
    pp = _fixture("intermediate_curvature")
    sol = hostsim.solve_kkt(pp, maxiter=2)
    assert sol["status"] != 0
    pbar, st = hostsim.sensitivity(pp, sol, np.ones(pp.layout.n), 1.0)
    assert st == CODES["skipped"] and (pbar == 0).all()
    # obstacle2d: the reduced Hessian at SLSQP's point is indefinite (DESIGN.md §4: down to -0.4 max|H|)
    pp = _fixture("obstacle2d")
    sol = hostsim.solve_kkt(pp)
    assert sol["status"] == 0
    pbar, st = hostsim.sensitivity(pp, sol, np.ones(pp.layout.n), 1.0)
    assert st == CODES["indefinite"] and (pbar == 0).all()
    # SLSQP's own point (stationarity ~1e-3) is inexact but carries values
    pp = _fixture("intermediate_curvature")
    sol = hostsim.solve_kkt(pp)
    assert sol["status"] == 0 and sol["kkt"][0] > 1e-6
    pbar, st = hostsim.sensitivity(pp, sol, np.ones(pp.layout.n), 1.0)
    assert st == CODES["inexact"] and np.abs(pbar).max() > 0 and np.isfinite(pbar).all()
    # a looser tolerance accepts it
    _, st = hostsim.sensitivity(pp, sol, np.ones(pp.layout.n), 1.0, tol=1.0)
    assert st in (CODES["ok"], CODES["nonstrict"])


def test_entry_points_fail_loudly_without_a_device(native_lib):
    import ctypes
    import torch
    from trajectory_generator_b200 import _native, batch, synthetic
    if torch.cuda.is_available():
        pytest.skip("a device is present")
    bt = synthetic.make("C2", 2)
    spec, sp = _native.spec_ptr(bt.spec)
    buf = (ctypes.c_double * 256)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    L = _native.lib()
    assert L.tg_sens_batch(sp, 2, *([p] * 8), 1e-6, None, 0, None) == 10
    assert b"no CUDA device" in L.tg_last_error()
    assert L.tg_sens_batch(sp, 2, None, *([p] * 7), 1e-6, None, 0, None) == 1
    assert L.tg_sens_workspace_bytes(sp, 2) == 0
    with pytest.raises(RuntimeError):
        batch.sensitivity_plan(bt.spec, 2)
    lay = bt.layout
    res = dict(x=torch.zeros(2, lay.n, dtype=torch.float64), f=torch.zeros(2, dtype=torch.float64),
               status=torch.zeros(2, dtype=torch.int32), lam=torch.zeros(2, lay.m, dtype=torch.float64))
    with pytest.raises(RuntimeError):
        batch.sensitivity(bt.spec, torch.from_numpy(bt.par), res, torch.zeros(2, lay.n, dtype=torch.float64))
    with pytest.raises(ValueError):
        batch.sensitivity(bt.spec, torch.from_numpy(bt.par), dict(x=res["x"], status=res["status"]),
                          torch.zeros(2, lay.n, dtype=torch.float64))
    with pytest.raises(RuntimeError):
        batch.solve_differentiable(bt.spec, torch.from_numpy(bt.par), torch.from_numpy(bt.x0))


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _np(out):
    return {k: (v.detach().cpu().numpy() if hasattr(v, "cpu") else v) for k, v in out.items() if k != "all"}


def _sens(spec, par, sol, x_bar, f_bar):
    """batch.sensitivity on device copies of numpy rows"""
    from trajectory_generator_b200 import batch
    rows = dict(x=_dev(sol["x"]), status=_dev(np.asarray(sol["status"], np.int32)), lam=_dev(sol["lam"]))
    return _np(batch.sensitivity(spec, _dev(par), rows, _dev(x_bar), None if f_bar is None else _dev(f_bar)))


def _bits(a, b):
    return np.array_equal(np.asarray(a).view(np.uint8), np.asarray(b).view(np.uint8))


@pytest.mark.gpu
def test_device_follows_host_build(native_lib, hostsim):
    """the device against the single-lane host build: the same status; par_bar within 1e-9 relative to max|par_bar|.
    (Not bit for bit: the device folds the objective's gradient sums across the lanes of a group and the host build
    sums on one lane; last-bit differences of g are amplified by the 1/h of the Hessian's central differences.)"""
    rng = np.random.default_rng(3)
    cases = [(n, pp, sol) for n, pp, sol in _stationary_cases(hostsim)]
    for name in ("obstacle2d", "intermediate_curvature"):
        pp = _fixture(name)
        cases.append((name + "/slsqp", pp, hostsim.solve_kkt(pp)))
    pp = _fixture("intermediate_curvature")
    cases.append(("iteration-limit", pp, hostsim.solve_kkt(pp, maxiter=2)))
    worst = 0.0
    for name, pp, sol in cases:
        x_bar, f_bar = rng.standard_normal(pp.layout.n), float(rng.standard_normal())
        ref, st = hostsim.sensitivity(pp, sol, x_bar, f_bar)
        out = _sens(pp.spec, pp.par[None], dict(x=sol["x"][None], status=[sol["status"]], lam=sol["lam"][None]),
                    x_bar[None], np.array([f_bar]))
        assert out["sens_status"][0] == st, (name, out["sens_status"][0], st)
        err = np.abs(out["par_bar"][0] - ref).max() / max(np.abs(ref).max(), 1e-300)
        worst = max(worst, err if np.abs(ref).max() > 0 else np.abs(out["par_bar"][0]).max())
        assert err <= 1e-9 if np.abs(ref).max() > 0 else (out["par_bar"][0] == 0).all(), (name, err)
    print("device vs host build: worst relative difference %.2e" % worst)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["C2", "C4"])
def test_positions_placements_and_instantiations_agree(native_lib, monkeypatch, name):
    from trajectory_generator_b200 import batch, synthetic
    bt = synthetic.make(name, 256)
    sol = _np(batch.solve(bt.spec, _dev(bt.par), _dev(bt.x0), jacobian="fd", polish=True))
    rng = np.random.default_rng(7)
    x_bar, f_bar = rng.standard_normal((256, bt.layout.n)), rng.standard_normal(256)
    base = _sens(bt.spec, bt.par, sol, x_bar, f_bar)
    assert (base["sens_status"] <= 1).sum() >= 64, np.bincount(base["sens_status"])
    perm = rng.permutation(256)
    shuf = _sens(bt.spec, bt.par[perm], {k: sol[k][perm] for k in ("x", "status", "lam")}, x_bar[perm], f_bar[perm])
    assert _bits(shuf["par_bar"], base["par_bar"][perm]) and _bits(shuf["sens_status"], base["sens_status"][perm])
    assert batch.sensitivity_plan(bt.spec, 256)["far"] == 0
    monkeypatch.setenv("TG_POLISH_FAR", "1")
    assert batch.sensitivity_plan(bt.spec, 256)["far"] == 1
    far = _sens(bt.spec, bt.par, sol, x_bar, f_bar)
    monkeypatch.delenv("TG_POLISH_FAR")
    monkeypatch.setenv("TG_GENERIC_KERNELS", "1")
    generic = _sens(bt.spec, bt.par, sol, x_bar, f_bar)
    monkeypatch.delenv("TG_GENERIC_KERNELS")
    for other in (far, generic):
        assert _bits(other["par_bar"], base["par_bar"]) and _bits(other["sens_status"], base["sens_status"])
    # f_bar = None is f_bar = 0
    nof = _sens(bt.spec, bt.par, sol, x_bar, None)
    assert _bits(nof["par_bar"], _sens(bt.spec, bt.par, sol, x_bar, np.zeros(256))["par_bar"])


@pytest.mark.gpu
def test_multistart_winner_equals_its_start_alone(native_lib):
    from trajectory_generator_b200 import batch, synthetic
    bt = synthetic.make("C2", 128)
    K = 4
    ms = _np(batch.solve_multistart(bt.spec, _dev(bt.par), _dev(bt.x0), K, seed=5, polish=True))
    par_x, x_x = batch.multistart_expand(bt.spec, _dev(bt.par), _dev(bt.x0), K, 5)
    rows = np.arange(128) * K + ms["best_start"]
    alone = _np(batch.solve(bt.spec, par_x[rows].contiguous(), x_x[rows].contiguous(), polish=True))
    rng = np.random.default_rng(9)
    x_bar, f_bar = rng.standard_normal((128, bt.layout.n)), rng.standard_normal(128)
    a = _sens(bt.spec, bt.par, ms, x_bar, f_bar)
    b = _sens(bt.spec, par_x[rows].cpu().numpy(), alone, x_bar, f_bar)
    assert _bits(a["par_bar"], b["par_bar"]) and _bits(a["sens_status"], b["sens_status"])


def _working_set(L, lam):
    return (np.arange(L.m)[None] < L.meq) | (lam > 0)


def _at_bound(L, x):
    xl = np.full(L.n, -np.inf); xu = np.full(L.n, np.inf)
    xl[L.ia:L.it0] = 10e-8
    if L.it0 < L.n:
        xl[L.it0:] = 0; xu[L.it0:] = L.N - 3
    return (x == xl) | (x == xu)


def _re_solve(spec, par, x_star, jacobian):
    """solve from x* (ftol 1e-12, maxiter 400, polished), then a second polish at tol 1e-12 (maxiter 20): the default
    polish tolerance (1e-8) leaves errors of x that the 1 / 2h of the comparison would amplify beyond 1e-4.  Returns the
    rows and a mask of those that are stationary to 1e-11 max(1, max|g|) with nonnegative inequality multipliers --
    tg_sens_batch's `inexact` test at tol 1e-11"""
    from trajectory_generator_b200 import batch
    P = _dev(par)
    r = batch.solve(spec, P, _dev(x_star), jacobian=jacobian, ftol=1e-12, maxiter=400, polish=True)
    batch.polish(spec, P, r, maxiter=20, tol=1e-12)
    st = batch.sensitivity(spec, P, r, r["x"].new_zeros(r["x"].shape), tol=1e-11)["sens_status"].cpu().numpy()
    r = _np(r)
    return r, (r["status"] == 0) & (st <= 1)


def _compare_with_re_solves(spec, L, par_at, sol, sens_status, x_bar, f_bar, an, jacobian, h=1e-5):
    """(x_bar . dx + f_bar df) / dt from re-solves at par_at(+-h) and par_at(+-h/2) against the analytic values `an`.
    A row is compared when its sensitivity is `ok`, its four re-solves are stationary (_re_solve) with the solve's
    working set and bound pattern, and the two difference quotients agree to 2e-5 (the response is linear at this
    scale: near a nearly singular reduced Hessian it is not, and the quotient measures curvature, not the derivative).
    Returns (compared mask, disagreeing mask)."""
    W, bnd = _working_set(L, sol["lam"]), _at_bound(L, sol["x"])
    keep = (sens_status == 0) & (sol["status"] == 0)
    fds = []
    for t in (h, h / 2):
        res = []
        for s in (1, -1):
            r, tight = _re_solve(spec, par_at(s * t), sol["x"], jacobian)
            keep &= tight & (_working_set(L, r["lam"]) == W).all(1) & (_at_bound(L, r["x"]) == bnd).all(1)
            res.append(r)
        fds.append((np.einsum("bn,bn->b", x_bar, res[0]["x"] - res[1]["x"]) + f_bar * (res[0]["f"] - res[1]["f"]))
                   / (2 * t))
    scale = np.maximum(np.maximum(np.abs(fds[0]), np.abs(an)), 1e-300)
    keep &= np.abs(fds[0] - fds[1]) <= 2e-5 * scale
    return keep, keep & ~(np.abs(fds[0] - an) <= 1e-4 * scale)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["C3", "C4"])
@pytest.mark.parametrize("jacobian", ["analytic", "fd"])
def test_against_re_solves(native_lib, name, jacobian):
    """<p_bar, delta> against re-solves from x* at par +- h delta (see _compare_with_re_solves): every compared row
    agrees to 1e-4 relative.  Compared on an NVIDIA B200: C3 41 (analytic) and 41 (fd) of 64 rows, C4 29 and 55; the
    others are rows whose re-solves change the working set or the bound pattern, or do not reach stationarity 1e-11,
    or whose response is not linear at h (a third of the rows is the floor asserted)"""
    from trajectory_generator_b200 import batch, synthetic
    B = 64
    bt = synthetic.make(name, B)
    L = bt.layout
    sol = _np(batch.solve(bt.spec, _dev(bt.par), _dev(bt.x0), jacobian=jacobian, polish=True))
    rng = np.random.default_rng(13)
    x_bar, f_bar = rng.standard_normal((B, L.n)), rng.standard_normal(B)
    sens = _sens(bt.spec, bt.par, sol, x_bar, f_bar)
    delta = rng.standard_normal((B, L.P)) * np.maximum(1.0, np.abs(bt.par))
    an = np.einsum("bp,bp->b", sens["par_bar"], delta)
    keep, bad = _compare_with_re_solves(bt.spec, L, lambda t: bt.par + t * delta, sol, sens["sens_status"], x_bar,
                                        f_bar, an, jacobian)
    print("%s %s: %d of %d rows compared, %d disagree; sens_status %s" % (
        name, jacobian, keep.sum(), B, bad.sum(), np.bincount(sens["sens_status"], minlength=7).tolist()))
    assert not bad.any(), np.flatnonzero(bad)
    assert keep.sum() >= B // 3


@pytest.mark.gpu
def test_solve_differentiable_forward_and_zero_rows(native_lib):
    import torch
    from trajectory_generator_b200 import batch, synthetic
    bt = synthetic.make("C2", 256)
    ref = _np(batch.solve(bt.spec, _dev(bt.par), _dev(bt.x0), multipliers=True, polish=True))
    par = _dev(bt.par).requires_grad_()
    x0 = _dev(bt.x0)
    x, f, res = batch.solve_differentiable(bt.spec, par, x0)
    assert _bits(x0.cpu().numpy(), bt.x0)                     # x0 is not modified
    out = _np(res)
    for k in ("x", "f", "status", "nit", "violation", "lam", "kkt", "polish_status", "polish_iters"):
        assert _bits(out[k], ref[k]), k
    assert x.requires_grad and f.requires_grad and not res["lam"].requires_grad
    w = torch.from_numpy(np.random.default_rng(1).standard_normal((256, bt.layout.n))).cuda()
    ((w * x).sum() + f.sum()).backward()
    g = par.grad.cpu().numpy()
    sens = _sens(bt.spec, bt.par, ref, w.cpu().numpy(), np.ones(256))
    assert _bits(g, sens["par_bar"])
    assert (g[ref["status"] != 0] == 0).all()
    assert (ref["status"] != 0).any()
    # only f used: x's gradient counts as zeros
    par2 = _dev(bt.par).requires_grad_()
    _, f2, _ = batch.solve_differentiable(bt.spec, par2, x0)
    f2.sum().backward()
    assert _bits(par2.grad.cpu().numpy(), _sens(bt.spec, bt.par, ref, np.zeros((256, bt.layout.n)), np.ones(256))["par_bar"])


def _c4_problem(b, start):
    from trajectory_generator_b200.batched import BatchedProblem
    r = b.raw
    p = r["points"]
    seglen = np.linalg.norm(p[:, :, 1:] - p[:, :, :-1], 2, 1)
    pad = r["dims"].copy(); pad[:, :, 0] -= seglen
    return BatchedProblem(3, start, _dev(p[:, :, 4]), _dev(r["v0"]), end_zero_velocity=True, max_velocity=r["vmax"],
                          max_acceleration=r["amax"], corridor_points=_dev(p), corridor_pads=_dev(pad),
                          objective_function_type="minimal_velocity_path")


@pytest.mark.gpu
def test_batched_problem_backward_reaches_the_start(native_lib):
    """C4 built by BatchedProblem with start.requires_grad_(): loss = (w x).sum() + f.sum(); start.grad against re-solves
    at start +- h delta (_compare_with_re_solves); a plain solve() is unchanged"""
    import torch
    from trajectory_generator_b200 import synthetic
    B = 64
    b = synthetic.make("C4", B)
    s0 = b.raw["points"][:, :, 0]
    plain = _np(_c4_problem(b, _dev(s0)).solve())
    s = _dev(s0).requires_grad_()
    bp = _c4_problem(b, s)
    out = bp.solve(differentiable=True)
    assert _bits(_np(bp.solve())["x"], plain["x"])
    L = bp.layout
    w = torch.from_numpy(np.random.default_rng(2).standard_normal((B, L.n))).cuda()
    ((w * out["x"]).sum() + out["f"].sum()).backward()
    grad = s.grad.cpu().numpy()
    o = _np(out)
    sens = _sens(bp.spec, bp.par.detach().cpu().numpy(), o, w.cpu().numpy(), np.ones(B))
    assert (grad[o["status"] != 0] == 0).all()
    delta = np.random.default_rng(4).standard_normal(s0.shape) * np.maximum(1.0, np.abs(s0))
    an = np.einsum("bd,bd->b", grad, delta)
    keep, bad = _compare_with_re_solves(bp.spec, L, lambda t: _c4_problem(b, _dev(s0 + t * delta)).par.detach().cpu().numpy(),
                                        o, sens["sens_status"], w.cpu().numpy(), np.ones(B), an, "fd")
    print("BatchedProblem C4: %d of %d rows compared, %d disagree" % (keep.sum(), B, bad.sum()))
    assert not bad.any(), np.flatnonzero(bad)
    assert keep.sum() >= B // 2
