"""KKT multipliers and the first-order optimality certificate of the batched solves (csrc/tg_sqp.h, tg_sqp_kkt;
batch.solve(..., multipliers=True); DESIGN.md §4 *Multipliers and the KKT certificate*).

CPU: the host build against scipy's compiled SLSQP core (its OptimizeResult.multipliers), against the full-space build
(-DTG_NO_ELIM, which forms every row's multiplier inside the QP), and the certificate's arithmetic against numpy.
GPU: bit-identity across batch sizes, placements, instantiations and entry points; the device against the host build
and against numpy from batch.evaluate + batch.linear_rows."""
import numpy as np
import pytest

import helpers
import hostsim_kkt
import problems
from trajectory_generator_b200.problem import Layout, pack_problem

CONVERGING = ["obstacle2d", "obstacles8", "intermediate_curvature", "sfc3d", "sfc3d_four"]


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


def _eliminated(L):
    """(rows the QP eliminates, whether they are pinned control points) -- the rule of tg_sqp_pinned"""
    d = L.d
    s = 3 if L.n_start == 3 * d else 1 if L.n_start == d else 0
    e = 3 if L.n_end == 3 * d else 1 if (L.n_end == d and L.p_sdir == L.p_target_vel) else 0
    if s == 3 or e == 3:
        s, e = (3 if s == 3 else 0), (3 if e == 3 else 0)
    rows = np.zeros(L.m, dtype=bool)
    if L.N >= 6:
        rows[L.r_start:L.r_start + s * d] = True
        rows[L.r_end:L.r_end + e * d] = True
    return rows, s == 3 or e == 3


def _kkt_numpy(L, xl, xu, x, g, c, J, lam):
    """the certificate restated: g, c, J (all m rows, dense) at x"""
    gl = g - J.T @ lam
    pi = np.where(x == xl, np.minimum(gl, 0), np.where(x == xu, np.maximum(gl, 0), gl))
    ineq = np.arange(L.m) >= L.meq
    fold = lambda v: np.inf if np.isnan(v).any() else (v.max() if v.size else 0.0)
    return np.array([fold(np.abs(pi)), max(fold(np.abs(c[~ineq])), fold(np.maximum(0, -c[ineq]))),
                     fold(np.maximum(0, -lam[ineq])), fold(np.abs(lam[ineq] * c[ineq]))]), \
        max(1.0, np.abs(g).max(), (np.abs(J) * np.abs(lam)[:, None]).sum(0).max())


@pytest.fixture(scope="module")
def hostsim():
    return hostsim_kkt.load()


@pytest.fixture(scope="module")
def full_space():
    return hostsim_kkt.load("noelim", ["-DTG_NO_ELIM"])


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
# Measured spread (max |lam - scipy| / max |lam_scipy|): rows the QP keeps 1e-14 ... 8e-11; eliminated rows of rotated
# location triples (obstacle2d, obstacles8, intermediate_curvature) 2e-14 ... 3e-10; pinned control points once the pins
# hold (sfc3d, sfc3d_four: the frozen block of the factor, DESIGN.md §4) 1.3e-5 and 3.6e-2.
@pytest.mark.parametrize("name", CONVERGING)
def test_multipliers_follow_scipy_slsqp_core(native_lib, hostsim, name):
    pp = _fixture(name)
    ref = hostsim_kkt.scipy_core_multipliers(hostsim, pp)
    mine = hostsim.solve_kkt(pp)
    assert (mine["status"], mine["nit"]) == (ref["status"], ref["nit"]) == (0, ref["nit"])
    assert np.abs(mine["x"] - ref["x"]).max() <= 1e-8
    rows, pinned = _eliminated(pp.layout)
    scale = np.abs(ref["multipliers"]).max()
    err = np.abs(mine["lam"] - ref["multipliers"]) / scale
    assert err[~rows].max() <= 1e-9
    assert err[rows].max() <= (0.1 if pinned else 1e-8)


def test_multipliers_follow_the_full_space_subproblem(native_lib, hostsim, full_space):
    """the recovery of the eliminated rows' multipliers against the build that keeps those rows in the QP, wherever both
    end in status 0 at the same x (measured: rotated triples <= 2.2e-9, pins that hold <= 3.6e-2 relative, the other
    rows <= 2.9e-9)"""
    cases = [(n, pp) for n in ("C2", "C3", "C4", "C5a") for pp in _synthetic(n, 8)] + \
            [(n, _fixture(n)) for n in problems.ALL]
    compared = {False: 0, True: 0}
    for name, pp in cases:
        a, b = hostsim.solve_kkt(pp), full_space.solve_kkt(pp)
        if not (a["status"] == b["status"] == 0 and np.abs(a["x"] - b["x"]).max() <= 1e-9):
            continue
        rows, pinned = _eliminated(pp.layout)
        err = np.abs(a["lam"] - b["lam"]) / max(1.0, np.abs(b["lam"]).max())
        assert err[~rows].max() <= 1e-8, name
        if rows.any():
            assert err[rows].max() <= (0.1 if pinned else 1e-8), name
            compared[pinned] += 1
    assert compared[False] >= 8 and compared[True] >= 4, compared


@pytest.mark.parametrize("jac", ["analytic", "fd"])
def test_certificate_arithmetic_and_signs(native_lib, hostsim, jac):
    """kkt equals its numpy restatement from hs.eval at the final x (analytic mode: the solver's own derivatives);
    inequality multipliers are >= 0 after every converged solve"""
    cases = [(n, _fixture(n)) for n in problems.ALL] + [(n, pp) for n in ("C2", "C4") for pp in _synthetic(n, 3)]
    for name, pp in cases:
        r = hostsim.solve_kkt(pp, fd=jac == "fd")
        L = pp.layout
        if r["status"] == 0:          # (a diverged solve -- features3d ends in exit 6 -- may certify inf)
            assert (r["lam"][L.meq:] >= 0).all() and r["kkt"][2] == 0, name
            assert np.isfinite(r["kkt"]).all(), name
        assert (r["kkt"] >= 0).all(), name
        if jac == "analytic":
            _, g, c, J = hostsim.eval(pp, r["x"])
            want, scale = _kkt_numpy(L, pp.xl, pp.xu, r["x"], g, c, J, r["lam"])
            assert abs(r["kkt"][0] - want[0]) <= 1e-12 * scale, name
            assert np.abs(r["kkt"][1:] - want[1:]).max() <= 1e-12 * max(1.0, np.abs(want[1:]).max()), name


def test_row_blocks_tile_the_rows(native_lib):
    from trajectory_generator_b200 import synthetic as syn
    specs = [_fixture(n).spec for n in problems.ALL] + [syn.make(n, 1).spec for n in ("C2", "C3", "C4", "C5a")]
    for spec in specs:
        L = Layout(spec)
        blocks = L.row_blocks()
        assert blocks[0][1] == 0 and blocks[-1][2] == L.m
        assert all(a[2] == b[1] for a, b in zip(blocks, blocks[1:]))
        assert all(b[1] < b[2] for b in blocks)
        eq = [b for b in blocks if b[3] == "eq"]
        assert eq and eq[-1][2] == L.meq and all(b[3] == "eq" for b in blocks[:len(eq)])


def test_entry_points_fail_without_device(native_lib):
    import ctypes

    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    from trajectory_generator_b200 import _native, batch, synthetic
    bt = synthetic.make("C2", 2)
    lay = bt.layout
    spec, sp = _native.spec_ptr(bt.spec)
    L = _native.lib()
    buf = np.zeros(64 * (lay.n + lay.P + lay.m))
    p = ctypes.c_void_p(buf.ctypes.data)
    assert L.tg_solve_batch_kkt(sp, 2, p, p, p, p, p, p, 100, 1e-6, 0, p, buf.nbytes, None, p, p) != 0
    assert L.tg_last_error().decode()
    L.tg_solve_mixed_batch_kkt.restype = ctypes.c_int
    ptrs = (ctypes.c_void_p * 1)(buf.ctypes.data)
    counts = np.array([2], dtype=np.int32)
    assert L.tg_solve_mixed_batch_kkt(1, spec.ctypes.data, counts.ctypes.data, ptrs, ptrs, ptrs, ptrs, ptrs, ptrs, 100,
                                      ctypes.c_double(1e-6), 0, None, ptrs, ptrs) != 0
    assert "no CUDA device" in L.tg_last_error().decode()
    with pytest.raises(RuntimeError, match="CUDA tensors"):
        batch.solve(bt.spec, torch.from_numpy(bt.par), torch.from_numpy(bt.x0), multipliers=True)


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _np(out):
    return {k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in out.items()}


def _same(a, b, keys):
    for k in keys:
        assert np.array_equal(np.asarray(a[k]).view(np.uint8), np.asarray(b[k]).view(np.uint8)), k


BASE = ("x", "f", "status", "nit", "violation")
KKT = ("lam", "kkt")


def _solve(bt, rows=None, **kw):
    from trajectory_generator_b200 import batch
    par, x0 = (bt.par, bt.x0) if rows is None else (bt.par[rows], bt.x0[rows])
    return _np(batch.solve(bt.spec, _dev(par), _dev(x0), **kw))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["C2", "C3", "C4", "C5a"])
@pytest.mark.parametrize("jacobian", ["analytic", "fd"])
def test_outputs_unchanged_and_positions_do_not_matter(native_lib, name, jacobian):
    from trajectory_generator_b200 import synthetic
    bt = synthetic.make(name, 1024)
    plain = _solve(bt, jacobian=jacobian)
    full = _solve(bt, jacobian=jacobian, multipliers=True)
    _same(plain, full, BASE)
    assert full["lam"].shape == (1024, bt.layout.m) and full["kkt"].shape == (1024, 4)
    for rows in (np.arange(1000, 1024), np.arange(512)[::-1], np.array([7])):
        part = _solve(bt, rows, jacobian=jacobian, multipliers=True)
        _same({k: full[k][rows] for k in BASE + KKT}, part, BASE + KKT)


@pytest.mark.gpu
def test_mixed_buckets_equal_single_solves(native_lib):
    from trajectory_generator_b200 import batch, synthetic
    bts = [synthetic.make(n, 300) for n in ("C2", "C4", "C3")]
    outs = batch.solve_mixed([(bt.spec, _dev(bt.par), _dev(bt.x0)) for bt in bts], multipliers=True)
    for bt, out in zip(bts, outs):
        _same(_np(out), _solve(bt, multipliers=True), BASE + KKT)


@pytest.mark.gpu
def test_placement_and_instantiation_do_not_matter(native_lib, monkeypatch):
    from trajectory_generator_b200 import synthetic
    bt = synthetic.make("C3", 256)
    monkeypatch.setenv("TG_QP_GS", "64")
    near = _solve(bt, multipliers=True)
    monkeypatch.setenv("TG_QP_FAR", "1")
    _same(near, _solve(bt, multipliers=True), BASE + KKT)
    monkeypatch.delenv("TG_QP_FAR"); monkeypatch.delenv("TG_QP_GS")
    c4 = synthetic.make("C4", 256)
    fixed = _solve(c4, multipliers=True, jacobian="fd")
    monkeypatch.setenv("TG_GENERIC_KERNELS", "1")
    _same(fixed, _solve(c4, multipliers=True, jacobian="fd"), BASE + KKT)


@pytest.mark.gpu
def test_multistart_gathers_the_winners_rows(native_lib):
    from trajectory_generator_b200 import batch, synthetic
    bt = synthetic.make("C2", 200)
    one = _np(batch.solve_multistart(bt.spec, _dev(bt.par), _dev(bt.x0), 1, multipliers=True))
    _same(one, _solve(bt, multipliers=True), BASE + KKT)
    K = 4
    ms = batch.solve_multistart(bt.spec, _dev(bt.par), _dev(bt.x0), K, seed=3, multipliers=True, return_all=True)
    allr = _np(ms.pop("all"))
    ms = _np(ms)
    par_x, x_x = batch.multistart_expand(bt.spec, _dev(bt.par), _dev(bt.x0), K, 3)
    ref = _np(batch.solve(bt.spec, par_x, x_x, multipliers=True))
    assert np.array_equal(allr["lam"].reshape(-1, bt.layout.m), ref["lam"])
    assert np.array_equal(allr["kkt"].reshape(-1, 4), ref["kkt"])
    rows = np.arange(200) * K + ms["best_start"]
    assert np.array_equal(ms["lam"], ref["lam"][rows]) and np.array_equal(ms["kkt"], ref["kkt"][rows])


@pytest.mark.gpu
def test_device_multipliers_follow_the_lock_step_host_build(native_lib):
    """the device stage is the host build's -DTG_FUSED_LM_FAR variant; where status and x agree within 1e-9 the
    multipliers agree to rounding (measured on the B200: see DESIGN.md §4)"""
    from trajectory_generator_b200 import batch
    far = hostsim_kkt.load("lmfar", ["-DTG_FUSED_LM_FAR"])
    compared = 0
    for name in problems.ALL:
        pp = _fixture(name)
        h = far.solve_kkt(pp)
        x0 = np.clip(pp.x0, pp.xl, pp.xu)[None]
        d = _np(batch.solve(pp.spec, _dev(pp.par[None]), _dev(x0), multipliers=True))
        if not (h["status"] == d["status"][0] and np.abs(h["x"] - d["x"][0]).max() <= 1e-9):
            continue
        assert np.abs(d["lam"][0] - h["lam"]).max() <= 1e-6 * max(1.0, np.abs(h["lam"]).max()), name
        compared += 1
    assert compared >= 5


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["C2", "C3", "C4", "C5a"])
def test_certificate_against_evaluate(native_lib, name):
    """kkt from numpy over batch.evaluate + batch.linear_rows + lam at the final x (analytic mode), to 1e-10 relative"""
    import torch
    from trajectory_generator_b200 import batch, synthetic
    bt = synthetic.make(name, 64)
    L = bt.layout
    out = _np(batch.solve(bt.spec, _dev(bt.par), _dev(bt.x0), multipliers=True))
    ev = _np(batch.evaluate(bt.spec, _dev(bt.par), _dev(out["x"])))
    A = batch.linear_rows(bt.spec, _dev(bt.par)).cpu().numpy()
    xl = np.full(L.n, -np.inf); xu = np.full(L.n, np.inf)
    xl[L.ia:L.it0] = 10e-8
    if L.it0 < L.n:
        xl[L.it0:] = 0; xu[L.it0:] = L.N - 3
    torch.cuda.synchronize()
    for b in range(64):
        J = A[b].copy()
        J[_nonlinear_rows(L)] = ev["jnl"][b]
        want, scale = _kkt_numpy(L, xl, xu, out["x"][b], ev["g"][b], ev["c"][b], J, out["lam"][b])
        assert abs(out["kkt"][b][0] - want[0]) <= 1e-10 * scale, b
        assert np.abs(out["kkt"][b][1:] - want[1:]).max() <= 1e-10 * max(1.0, np.abs(want[1:]).max()), b


def _nonlinear_rows(L):
    """rows whose Jacobian batch.evaluate returns in jnl (everything that tg_linear_rows_batch leaves zero)"""
    rows = np.zeros(L.m, dtype=bool)
    rows[L.r_sder:L.meq] = True
    rows[L.r_db:L.r_sfcl] = True
    rows[L.r_obs:L.r_obs + L.n_obs] = True
    return np.nonzero(rows)[0]


@pytest.mark.gpu
@pytest.mark.parametrize("fused", [False, True])
def test_long_shapes_give_a_finite_certificate(native_lib, fused):
    import test_large_shapes
    from trajectory_generator_b200 import batch
    for name in ("corridors8_3d", "waypoints3d", "extreme3d"):
        pp = test_large_shapes._packed(name)
        L = pp.layout
        x0 = np.repeat(np.clip(pp.x0, pp.xl, pp.xu)[None], 2, axis=0)
        out = _np(batch.solve(pp.spec, _dev(np.repeat(pp.par[None], 2, axis=0)), _dev(x0),
                              maxiter=test_large_shapes.MAXITER[name], fused=fused, multipliers=True))
        ok = out["status"] == 0
        assert ok.any() and np.isfinite(out["lam"]).all(), name
        assert np.isfinite(out["kkt"][ok]).all() and (out["lam"][ok][:, L.meq:] >= 0).all(), name


@pytest.mark.gpu
def test_dropin_class_gives_the_batch_multipliers(native_lib):
    from trajectory_generator_b200 import batch
    from trajectory_generator_b200.trajectory_generator import TrajectoryGenerator
    ns = helpers.product_namespace()
    names = [n for n in problems.ALL if problems.ALL[n](ns)[0] == 2][:4]
    ccs = [problems.ALL[n](ns) for n in names]
    tg = TrajectoryGenerator(2, jacobian="analytic", multipliers=True)
    default = TrajectoryGenerator(2, jacobian="analytic")
    for (d, cc, kw), name in zip(ccs, names):
        obj = kw.get("objective_function_type", "minimal_velocity_and_time_path")
        res = tg.generate_trajectories([cc], obj, kw.get("num_intervals_free_space"))[0]
        assert default.generate_trajectories([cc], obj, kw.get("num_intervals_free_space"))[0].multipliers is None
        pp = pack_problem(d, cc, obj, kw.get("num_intervals_free_space"))
        x0 = np.clip(pp.x0, pp.xl, pp.xu)[None]
        ref = _np(batch.solve(pp.spec, _dev(pp.par[None]), _dev(x0), multipliers=True))
        assert np.array_equal(res.multipliers, ref["lam"][0]) and np.array_equal(res.kkt, ref["kkt"][0]), name
        assert np.array_equal(res.x, ref["x"][0])
