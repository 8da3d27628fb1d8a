"""Post-solve polish (csrc/tg_polish.h, tg_polish_batch; batch.polish and the solve entry points' polish=True;
DESIGN.md §4 *Polish*).

CPU: the host build against a numpy restatement of the algorithm, the final guard, untouched rows, stationarity on the
converging fixtures, an independent check of kkt[0] with central differences of the oracle's numpy closures, and the
error paths without a device.
GPU: polish=False changes nothing; the device against the host build; bit-identity across batch positions, entry
points, placements, instantiations and multi-start; the guard against a recomputation from batch.evaluate; long
far-placed shapes; the drop-in class."""
import numpy as np
import pytest

import helpers
import hostsim_polish
import problems
from trajectory_generator_b200.problem import pack_problem

MAXITER, TOL = 8, 1e-8
CONVERGING = ["obstacle2d", "obstacles8", "intermediate_curvature", "sfc3d", "sfc3d_four"]
REPLACED = (0, 1)           # polished, improved


def _fixture(name):
    d, cc, kw = problems.ALL[name](helpers.product_namespace())
    return pack_problem(d, cc, kw.get("objective_function_type", "minimal_velocity_and_time_path"),
                        kw.get("num_intervals_free_space"))


class _P:
    pass


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


def _cases():
    return [(n, _fixture(n)) for n in problems.ALL] + [(n, pp) for n in ("C2", "C4", "C5a") for pp in _synthetic(n, 3)]


@pytest.fixture(scope="module")
def hostsim():
    return hostsim_polish.load()


def _bounds(pp):
    return np.where(np.isfinite(pp.xl), pp.xl, -np.inf), np.where(np.isfinite(pp.xu), pp.xu, np.inf)


def _viol(L, c):
    return np.concatenate([np.abs(c[:L.meq]), np.maximum(-c[L.meq:], 0)])


def _stationarity(L, xl, xu, x, g, J, lam):
    gl = g - J.T @ lam
    pi = np.where(x == xl, np.minimum(gl, 0), np.where(x == xu, np.maximum(gl, 0), gl))
    return np.abs(pi).max()


def _restated(hs, pp, sol, maxiter=MAXITER, tol=TOL):
    """tg_polish_problem restated in numpy with f, g, c, J from HostSim.eval: (x, lam, status) of the polished point"""
    L = pp.layout
    n, m, meq = L.n, L.m, L.meq
    xl, xu = _bounds(pp)
    nl = np.array([not (L.r_start <= r < L.r_end + L.n_end or L.r_sfcl <= r < L.r_sfcu + L.n_sfc) for r in range(m)])
    x, lam = sol["x"].copy(), sol["lam"].copy()
    rho = 1 + 2 * np.abs(lam).max(initial=0)
    f, g, c, J = hs.eval(pp, x)
    merit = f + rho * _viol(L, c).sum()
    st = _stationarity(L, xl, xu, x, g, J, lam)
    it, drop, moved = 0, np.zeros(m, bool), False
    while True:
        if st <= tol * max(1.0, np.abs(g).max()):
            return x, lam, "polished", it, moved
        if it >= maxiter:
            return x, lam, "maxiter", it, moved
        free = np.flatnonzero((x != xl) & (x != xu))
        W = np.flatnonzero((np.arange(m) < meq) | ((lam > 0) & ~drop))
        if len(W) > len(free):
            return x, lam, "degenerate", it, moved
        H = np.zeros((len(free), len(free)))
        for b, i in enumerate(free):
            h = 6.0554544523933395e-06 * max(1.0, abs(x[i]))
            xp, xm = min(x[i] + h, xu[i]), max(x[i] - h, xl[i])
            cols = []
            for xv in (xp, xm):
                y = x.copy(); y[i] = xv
                _, gy, _, Jy = hs.eval(pp, y)
                cols.append(gy[free] - (Jy[nl].T @ lam[nl])[free])
            H[:, b] = (cols[0] - cols[1]) / (xp - xm)
        H = 0.5 * (H + H.T)
        A = J[np.ix_(W, free)]
        Q, R = np.linalg.qr(A.T, mode="complete")
        if (np.abs(np.diag(R)) < 1e-12 * np.abs(R).max(initial=0)).any():
            return x, lam, "degenerate", it, moved
        k = len(W)
        Y, Z = Q[:, :k], Q[:, k:]
        py = np.linalg.solve(R[:k].T, -c[W])
        Hz = Z.T @ H @ Z
        hmax = np.abs(H).max(initial=0)
        for delta in (0.0, 1e-8 * hmax, 1e-6 * hmax, 1e-4 * hmax):
            try:
                np.linalg.cholesky(Hz + delta * np.eye(len(Hz)))
                break
            except np.linalg.LinAlgError:
                delta = None
        if delta is None:
            return x, lam, "stalled", it, moved
        pz = np.linalg.solve(Hz + delta * np.eye(len(Hz)), -Z.T @ (g[free] + H @ (Y @ py)))
        p = Y @ py + Z @ pz
        lw = np.linalg.solve(R[:k], Y.T @ (g[free] + H @ p))
        neg = [(lw[q], W[q]) for q in range(k) if W[q] >= meq and lw[q] < 0]
        if neg:
            drop[min(neg)[1]] = True
            it += 1
            continue
        it += 1
        for a in (1.0, 0.5, 0.25, 0.125):
            xt = x.copy(); xt[free] = np.clip(x[free] + a * p, xl[free], xu[free])
            ft, _, ct, _ = hs.eval(pp, xt, jac=False)
            if ft + rho * _viol(L, ct).sum() <= merit:
                break
        else:
            return x, lam, "stalled", it, moved
        x, moved, drop[:] = xt, True, False
        lam = np.zeros(m); lam[W] = lw
        f, g, c, J = hs.eval(pp, x)
        merit = f + rho * _viol(L, c).sum()
        st = _stationarity(L, xl, xu, x, g, J, lam)


def _guard(hs, pp, sol, out):
    """the final guard from HostSim.eval at the input and the output points"""
    L = pp.layout
    xl, xu = _bounds(pp)
    rho = 1 + 2 * np.abs(sol["lam"]).max(initial=0)
    f0, g0, c0, J0 = hs.eval(pp, sol["x"])
    f1, g1, c1, J1 = hs.eval(pp, out["x"])
    assert np.isfinite(out["x"]).all() and np.isfinite(out["lam"]).all() and np.isfinite(out["kkt"]).all()
    assert _viol(L, c1).max(initial=0) <= max(_viol(L, c0).max(initial=0), 1e-8)
    assert f1 + rho * _viol(L, c1).sum() <= (f0 + rho * _viol(L, c0).sum()) * (1 + 1e-15) + 1e-300
    st0 = _stationarity(L, xl, xu, sol["x"], g0, J0, sol["lam"])
    st1 = _stationarity(L, xl, xu, out["x"], g1, J1, out["lam"])
    assert st1 < st0
    assert (out["lam"][L.meq:] >= -1e-8 * max(1.0, np.abs(out["lam"]).max())).all()
    return st0, st1


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def test_host_polish_follows_numpy_restatement(native_lib, hostsim):
    compared = 0
    for name, pp in _cases():
        sol = hostsim.solve_kkt(pp)
        out = hostsim.polish(pp, sol)
        x, lam, why, it, moved = _restated(hostsim, pp, sol)
        if sol["status"] != 0:
            assert out["polish_status"] == 4, name
            continue
        if why == "degenerate":
            assert out["polish_status"] == 3, name
            continue
        # (at the floor of the arithmetic -- stationarity ~1e-9 -- whether `tol` is met depends on the summation order of
        # gradL, numpy's against the serial sums: one more Newton step of size ~1e-12 on either side)
        assert abs(out["polish_iters"] - it) <= 1, (name, out["polish_iters"], it, why)
        if out["polish_status"] in REPLACED:
            # (1e-10 relative with the same iterations; one floor step more or less moves x by ~1e-9)
            rel = 1e-10 if out["polish_iters"] == it else 1e-9
            assert np.abs(out["x"] - x).max() <= rel * max(1.0, np.abs(x).max()), name
            assert np.abs(out["lam"] - lam).max() <= 1e-8 * max(1.0, np.abs(lam).max()), name
            compared += 1
    assert compared >= 6, compared


@pytest.mark.parametrize("jac", ["analytic", "fd"])
def test_guard_holds_and_untouched_rows_keep_their_bits(native_lib, hostsim, jac):
    counts = {}
    for name, pp in _cases():
        sol = hostsim.solve_kkt(pp, fd=jac == "fd")
        sol["violation"] = 0
        out = hostsim.polish(pp, sol)
        ps = out["polish_status"]
        counts[ps] = counts.get(ps, 0) + 1
        if ps in REPLACED:
            _guard(hostsim, pp, sol, out)
        else:
            for k in ("x", "lam", "kkt"):
                assert np.array_equal(out[k].view(np.uint8), np.asarray(sol[k], np.float64).view(np.uint8)), (name, k)
            assert out["f"] == sol["f"] or (np.isnan(out["f"]) and np.isnan(sol["f"]))
        # a row with status != 0 is skipped
        skipped = hostsim.polish(pp, dict(sol, status=1))
        assert skipped["polish_status"] == 4 and skipped["polish_iters"] == 0
        assert np.array_equal(skipped["x"], sol["x"]) and np.array_equal(skipped["lam"], sol["lam"])
    assert counts.get(0, 0) + counts.get(1, 0) >= 6, counts


# Stationarity on the converging fixtures (tol 1e-8 relative to max(1, max|g|)).  Not reached, recorded: obstacle2d,
# obstacles8 and sfc3d -- at SLSQP's point the reduced Hessian Z'HZ of the working set has eigenvalues down to -0.4
# max|H| (obstacle2d: -1.9e4 against max|H| = 4.3e4), beyond the regularisation ladder's 1e-4 max|H|: no Newton step,
# the row is returned as it was (rejected, 0 iterations).
STATIONARY = {"obstacle2d": False, "obstacles8": False, "intermediate_curvature": True, "sfc3d": False, "sfc3d_four": True}


@pytest.mark.parametrize("name", CONVERGING)
def test_converging_fixtures_become_stationary(native_lib, hostsim, name):
    pp = _fixture(name)
    sol = hostsim.solve_kkt(pp)
    out = hostsim.polish(pp, sol)
    _, g, _, _ = hostsim.eval(pp, out["x"])
    if not STATIONARY[name]:
        assert (out["polish_status"], out["polish_iters"]) == (2, 0)
        assert np.array_equal(out["x"], sol["x"])
        return
    assert out["polish_status"] == 0, (out["polish_status"], out["polish_iters"], out["kkt"][0], sol["kkt"][0])
    assert out["kkt"][0] <= TOL * max(1.0, np.abs(g).max())


def test_stationarity_against_oracle_closures(native_lib, hostsim):
    """kkt[0] of a polished row from central differences of the oracle's numpy closures (OracleProblem.fun / cons) and
    the returned multipliers, independently of the CUDA source: agreement to 1e-5 relative to max(1, max|g|) (the
    differences' truncation and rounding error at h = 1e-6)"""
    import tg_oracle
    checked = 0
    for name in problems.SOLVE:
        d, cc, kw = problems.ALL[name](helpers.product_namespace())
        pp = _fixture(name)
        op = tg_oracle.OracleProblem(d, cc, kw.get("objective_function_type", "minimal_velocity_and_time_path"),
                                     kw.get("num_intervals_free_space"))
        out = hostsim.polish(pp, hostsim.solve_kkt(pp))
        if out["polish_status"] not in REPLACED:
            continue
        x, L = out["x"], pp.layout
        h = 1e-6
        g = np.zeros(L.n); J = np.zeros((L.m, L.n))
        for i in range(L.n):
            e = np.zeros(L.n); e[i] = h * max(1.0, abs(x[i]))
            g[i] = (op.fun(x + e) - op.fun(x - e)) / (2 * e[i])
            J[:, i] = (np.asarray(op.cons(x + e)) - np.asarray(op.cons(x - e))) / (2 * e[i])
        xl, xu = _bounds(pp)
        st = _stationarity(L, xl, xu, x, g, J, out["lam"])
        assert abs(st - out["kkt"][0]) <= 1e-5 * max(1.0, np.abs(g).max()), (name, st, out["kkt"][0])
        checked += 1
    assert checked >= 1


def test_entry_points_fail_loudly_without_a_device(native_lib):
    import ctypes
    import torch
    from trajectory_generator_b200 import _native, batch, synthetic
    if torch.cuda.is_available():
        pytest.skip("a device is present")
    bt = synthetic.make("C2", 2)
    spec, sp = _native.spec_ptr(bt.spec)
    buf = (ctypes.c_double * 64)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    L = _native.lib()
    assert L.tg_polish_batch(sp, 2, *([p] * 9), 8, 1e-8, None, 0, None) == 10
    assert b"no CUDA device" in L.tg_last_error()
    assert L.tg_polish_batch(sp, 2, None, *([p] * 8), 8, 1e-8, None, 0, None) == 1
    assert L.tg_polish_workspace_bytes(sp, 2) == 0
    with pytest.raises(RuntimeError):
        batch.polish_plan(bt.spec, 2)
    res = dict(x=torch.zeros(2, bt.layout.n, dtype=torch.float64), lam=torch.zeros(2, bt.layout.m), kkt=torch.zeros(2, 4))
    with pytest.raises(RuntimeError):
        batch.polish(bt.spec, torch.from_numpy(bt.par), res)
    with pytest.raises(ValueError):
        batch.polish(bt.spec, torch.from_numpy(bt.par), dict(x=res["x"]))


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _np(out):
    return {k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in out.items() if k != "all"}


def _same(a, b, keys):
    for k in keys:
        assert np.array_equal(np.asarray(a[k]).view(np.uint8), np.asarray(b[k]).view(np.uint8)), k


BASE = ("x", "f", "status", "nit", "violation")
OUT = BASE + ("lam", "kkt", "polish_status", "polish_iters")


def _solve(bt, rows=None, **kw):
    from trajectory_generator_b200 import batch
    par, x0 = (bt.par, bt.x0) if rows is None else (bt.par[rows], bt.x0[rows])
    return _np(batch.solve(bt.spec, _dev(par), _dev(x0), **kw))


def _polish_copy(spec, par, sol, **kw):
    """batch.polish on device copies of a solve's numpy result"""
    from trajectory_generator_b200 import batch
    res = {k: _dev(sol[k]) for k in BASE + ("lam", "kkt")}
    return _np(batch.polish(spec, _dev(par), res, **kw))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["C2", "C3", "C4", "C5a"])
@pytest.mark.parametrize("jacobian", ["analytic", "fd"])
def test_polish_false_changes_nothing_and_positions_do_not_matter(native_lib, name, jacobian):
    from trajectory_generator_b200 import synthetic
    bt = synthetic.make(name, 512)
    plain = _solve(bt, jacobian=jacobian, multipliers=True)
    _same(plain, _solve(bt, jacobian=jacobian, multipliers=True, polish=False), BASE + ("lam", "kkt"))
    full = _solve(bt, jacobian=jacobian, polish=True)
    _same(plain, full, ("status", "nit"))
    for rows in (np.arange(500, 512), np.arange(256)[::-1], np.array([7])):
        part = _solve(bt, rows, jacobian=jacobian, polish=True)
        _same({k: full[k][rows] for k in OUT}, part, OUT)


@pytest.mark.gpu
def test_device_follows_host_build(native_lib, hostsim):
    """the device against the single-lane host build on the fixtures and synthetic problems: the same status, iterations
    within one, x within 1e-9 relative (the device folds the objective's value across the lanes of a group and the host
    build sums it on one lane: f differs in its last bits, and so may the arithmetic floor at which `tol` is met)"""
    compared = 0
    for name, pp in _cases():
        sol = hostsim.solve_kkt(pp)
        ref = hostsim.polish(pp, dict(sol, violation=0))
        rows = dict(x=sol["x"][None], f=np.array([sol["f"]]), status=np.array([sol["status"]], np.int32),
                    nit=np.array([sol["nit"]], np.int32), violation=np.zeros(1, np.int32), lam=sol["lam"][None],
                    kkt=sol["kkt"][None])
        out = _polish_copy(pp.spec, pp.par[None], rows)
        assert out["polish_status"][0] == ref["polish_status"], name
        assert abs(int(out["polish_iters"][0]) - ref["polish_iters"]) <= 1, name
        assert np.abs(out["x"][0] - ref["x"]).max() <= 1e-9 * max(1.0, np.abs(ref["x"]).max()), name
        compared += ref["polish_status"] in REPLACED
    assert compared >= 4


@pytest.mark.gpu
def test_entry_points_placements_and_instantiations_agree(native_lib, monkeypatch):
    from trajectory_generator_b200 import batch, synthetic
    bts = [synthetic.make(n, 200) for n in ("C2", "C4", "C3")]
    outs = [_np(o) for o in batch.solve_mixed([(bt.spec, _dev(bt.par), _dev(bt.x0)) for bt in bts], polish=True)]
    for bt, out in zip(bts, outs):
        _same(out, _solve(bt, polish=True), OUT)
    for bt in bts:
        sol = _solve(bt, multipliers=True, jacobian="fd")
        near = _polish_copy(bt.spec, bt.par, sol)
        assert batch.polish_plan(bt.spec, 200)["far"] == 0
        monkeypatch.setenv("TG_POLISH_FAR", "1")
        assert batch.polish_plan(bt.spec, 200)["far"] == 1
        _same(near, _polish_copy(bt.spec, bt.par, sol), OUT)
        monkeypatch.delenv("TG_POLISH_FAR")
        monkeypatch.setenv("TG_GENERIC_KERNELS", "1")
        _same(near, _polish_copy(bt.spec, bt.par, sol), OUT)
        monkeypatch.delenv("TG_GENERIC_KERNELS")


@pytest.mark.gpu
def test_multistart_winner_equals_its_start_polished_alone(native_lib):
    from trajectory_generator_b200 import batch, synthetic
    bt = synthetic.make("C2", 128)
    K = 4
    ms = batch.solve_multistart(bt.spec, _dev(bt.par), _dev(bt.x0), K, seed=5, polish=True, return_all=True)
    raw = _np(ms.pop("all"))
    ms = _np(ms)
    par_x, x_x = batch.multistart_expand(bt.spec, _dev(bt.par), _dev(bt.x0), K, 5)
    rows = np.arange(128) * K + ms["best_start"]
    alone = _np(batch.solve(bt.spec, par_x[rows].contiguous(), x_x[rows].contiguous(), polish=True))
    _same(ms, alone, OUT)
    plain = _np(batch.solve(bt.spec, par_x, x_x, multipliers=True))
    assert np.array_equal(raw["x"].reshape(-1, bt.layout.n), plain["x"])      # return_all rows stay raw
    assert np.array_equal(raw["lam"].reshape(-1, bt.layout.m), plain["lam"])
    rep = ms["polish_status"] <= 1
    assert np.array_equal(ms["max_violation"][rep], ms["kkt"][rep, 1])


def _recompute(bt, x, lam):
    """stationarity, max violation, merit parts from batch.evaluate + batch.linear_rows (analytic derivatives)"""
    import torch
    from trajectory_generator_b200 import batch
    L = bt.layout
    par = _dev(bt.par)
    ev = batch.evaluate(bt.spec, par, _dev(x))
    J = batch.linear_rows(bt.spec, par).cpu().numpy()
    lin = np.array([L.r_start <= r < L.r_end + L.n_end or L.r_sfcl <= r < L.r_sfcu + L.n_sfc for r in range(L.m)])
    J[:, ~lin, :] = ev["jnl"].cpu().numpy()
    g, c = ev["g"].cpu().numpy(), ev["c"].cpu().numpy()
    gl = g - np.einsum("bmn,bm->bn", J, lam)
    xl = np.full(L.n, -np.inf); xu = np.full(L.n, np.inf)
    xl[L.ia:L.it0] = 10e-8
    if L.it0 < L.n:
        xl[L.it0:] = 0; xu[L.it0:] = L.N - 3
    pi = np.where(x == xl, np.minimum(gl, 0), np.where(x == xu, np.maximum(gl, 0), gl))
    v = np.concatenate([np.abs(c[:, :L.meq]), np.maximum(-c[:, L.meq:], 0)], 1)
    return np.abs(pi).max(1), v.max(1, initial=0), ev["f"].cpu().numpy(), v.sum(1), np.abs(g).max(1)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["C2", "C3", "C4", "C5a"])
def test_guard_against_batch_evaluate(native_lib, name):
    from trajectory_generator_b200 import synthetic
    bt = synthetic.make(name, 4096)
    sol = _solve(bt, multipliers=True)
    out = _polish_copy(bt.spec, bt.par, sol)
    ok = sol["status"] == 0
    assert (out["polish_status"][~ok] == 4).all()
    st0, v0, f0, s0, g0 = _recompute(bt, sol["x"], sol["lam"])
    st1, v1, f1, s1, g1 = _recompute(bt, out["x"], out["lam"])
    rep = np.isin(out["polish_status"], REPLACED)
    rho = 1 + 2 * np.abs(sol["lam"]).max(1)
    scale = np.maximum(1.0, g0)
    assert (st1[ok] <= st0[ok] + 1e-9 * scale[ok]).all()             # no row's stationarity rises
    assert (st1[rep] < st0[rep] + 1e-12 * scale[rep]).all()
    assert (v1[rep] <= np.maximum(v0[rep], 1e-8) * (1 + 1e-9)).all()
    m0, m1 = f0 + rho * s0, f1 + rho * s1
    assert (m1[rep] <= m0[rep] + 1e-12 * np.maximum(1.0, np.abs(m0[rep]))).all()
    for k in ("x", "lam", "kkt", "f", "violation"):
        assert np.array_equal(out[k][~rep].view(np.uint8), sol[k][~rep].view(np.uint8)), k
    assert np.isfinite(out["x"][rep]).all() and np.isfinite(out["kkt"][rep]).all()
    # kkt[0] of a replaced row: the device's own stationarity from the same derivatives
    assert (np.abs(out["kkt"][rep, 0] - st1[rep]) <= 1e-9 * scale[rep]).all()


@pytest.mark.gpu
def test_long_far_placed_shapes_give_finite_results(native_lib):
    import torch
    import test_large_shapes as tls
    from trajectory_generator_b200 import batch
    cases = [(_fixture("long2d"), 100)] + [(tls._packed(n), tls.MAXITER[n]) for n in tls.LARGE]
    far = 0
    for pp, maxiter in cases:
        x0 = np.clip(pp.x0, pp.xl, pp.xu)[None]
        res = batch.solve(pp.spec, _dev(pp.par[None]), _dev(x0), maxiter=maxiter, polish=True)
        torch.cuda.synchronize()
        out = _np(res)
        far += batch.polish_plan(pp.spec, 1)["far"]
        if out["status"][0] == 0:
            assert out["polish_status"][0] != 4
            assert np.isfinite(out["x"]).all() and np.isfinite(out["kkt"]).all() and np.isfinite(out["lam"]).all()
    assert far >= 1


@pytest.mark.gpu
def test_dropin_class_returns_the_polished_rows(native_lib):
    from trajectory_generator_b200 import batch
    from trajectory_generator_b200.trajectory_generator import TrajectoryGenerator
    ns = helpers.product_namespace()
    gen = TrajectoryGenerator(2, jacobian="analytic", polish=True)
    for name in ["obstacle2d", "obstacles8", "intermediate_curvature"]:
        d, cc, kw = problems.ALL[name](ns)
        obj = kw.get("objective_function_type", "minimal_velocity_and_time_path")
        r = gen.generate_trajectories([cc], obj, kw.get("num_intervals_free_space"))[0]
        pp = pack_problem(d, cc, obj, kw.get("num_intervals_free_space"))
        x0 = np.clip(pp.x0, pp.xl, pp.xu)[None]
        ref = _np(batch.solve(pp.spec, _dev(pp.par[None]), _dev(x0), polish=True))
        assert np.array_equal(r.x, ref["x"][0]) and np.array_equal(r.multipliers, ref["lam"][0]), name
        assert np.array_equal(r.kkt, ref["kkt"][0]) and r.polish_status == int(ref["polish_status"][0]), name
