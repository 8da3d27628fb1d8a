"""Shapes whose QP scratch (and, for the largest, the line-search stage's share) does not fit in shared memory: the solve
places that scratch in per-lane-group slots of the workspace instead.  The fixtures are long trajectories of the kinds
users build (a corridor path of eight uneven corridors, a multi-waypoint mission); they are not part of problems.ALL,
which holds fixtures with recorded reference solves."""
import os

import numpy as np
import pytest

import helpers
import hostsim_loader
import problems

_col = problems._col
PTS8 = [_col(0, 0, 0), _col(5, 1, 1), _col(9, 6, 2), _col(24, 9, 5), _col(28, 13, 4), _col(31, 16, 6),
        _col(47, 21, 8), _col(50, 25, 9), _col(62, 31, 13)]


def corridors8_3d(ns, pts=PTS8, intervals_per_corridor=None):
    """Eight uneven corridors, intervals per corridor from the segment lengths (min 2): N = 49, n = 148."""
    W, WD, DB = ns["Waypoint"], ns["WaypointData"], ns["DerivativeBounds"]
    sfcs = []
    for i in range(len(pts) - 1):
        R, T, L = ns["get3DRotationAndTranslationFromPoints"](pts[i], pts[i + 1])
        sfcs.append(ns["SFC"](np.array([[L + 2.5], [2.4], [2.8]]), T, R))
    if intervals_per_corridor is None:
        sfc = ns["SFC_Data"](tuple(sfcs), np.concatenate(pts, 1), 2)
    else:
        sfc = ns["SFC_Data"](tuple(sfcs), np.concatenate(pts, 1), 2, intervals_per_corridor=np.array(intervals_per_corridor))
    v0 = (pts[1] - pts[0]) / np.linalg.norm(pts[1] - pts[0])
    wd = WD((W(location=pts[0], velocity=v0), W(location=pts[-1], velocity=_col(0, 0, 0))))
    cc = ns["ConstraintsContainer"](waypoint_constraints=wd, derivative_constraints=DB(5, 0.3), sfc_constraints=sfc)
    return 3, cc, dict(objective_function_type="minimal_velocity_path")


def waypoints3d(ns, shift=None):
    """A mission through three intermediate waypoints around two spheres, 36 intervals: N = 39, n = 121."""
    W, WD, DB, TB, Ob = ns["Waypoint"], ns["WaypointData"], ns["DerivativeBounds"], ns["TurningBound"], ns["Obstacle"]
    locs = [(0, 0, 0), (6, 4, 1), (10, 10, 3), (14, 12, 2), (20, 18, 4)]
    if shift is not None:
        locs = [locs[0]] + [tuple(np.add(p, s)) for p, s in zip(locs[1:4], shift)] + [locs[4]]
    seq = (W(location=_col(*locs[0]), velocity=_col(1, 0, 0)),) + tuple(W(location=_col(*p)) for p in locs[1:4]) + \
          (W(location=_col(*locs[4]), velocity=_col(0, 1, 0)),)
    obs = [Ob(center=_col(3, 2, 0.5), radius=0.8), Ob(center=_col(12, 11, 2.5), radius=0.7)]
    cc = ns["ConstraintsContainer"](waypoint_constraints=WD(seq), derivative_constraints=DB(4, 3),
                                    turning_constraint=TB(2, "angular_rate"), obstacle_constraints=obs)
    return 3, cc, dict(objective_function_type="minimal_velocity_path", num_intervals_free_space=36)


def extreme3d(ns):
    """corridors8_3d with 15 intervals in every corridor: N = 123, n = 370 (the line-search stage's share does not fit
    either)."""
    return corridors8_3d(ns, intervals_per_corridor=[15] * 8)


LARGE = dict(corridors8_3d=corridors8_3d, waypoints3d=waypoints3d, extreme3d=extreme3d)
MAXITER = dict(corridors8_3d=500, waypoints3d=500, extreme3d=1000)


def _packed(name, fixture=None):
    from trajectory_generator_b200.problem import pack_problem
    d, cc, kw = (fixture or LARGE[name])(helpers.product_namespace())
    return pack_problem(d, cc, kw.get("objective_function_type", "minimal_velocity_and_time_path"),
                        kw.get("num_intervals_free_space"))


def _perturbed(name, count, seed):
    """`count` copies of a fixture with its corridor points / intermediate waypoints moved by up to +-0.3, all of the
    fixture's shape (copies whose interval rule picks another shape are skipped): (spec, par [B, P], x0 [B, n])."""
    from trajectory_generator_b200.problem import pack_problem
    ns = helpers.product_namespace()
    base = _packed(name)
    rng = np.random.default_rng(seed)
    pars, xs = [], []
    while len(pars) < count:
        if name == "waypoints3d":
            d, cc, kw = waypoints3d(ns, shift=rng.uniform(-0.3, 0.3, (3, 3)))
        else:
            pts = [PTS8[0]] + [p + rng.uniform(-0.3, 0.3, (3, 1)) for p in PTS8[1:-1]] + [PTS8[-1]]
            d, cc, kw = corridors8_3d(ns, pts=pts)
        pp = pack_problem(d, cc, kw["objective_function_type"], kw.get("num_intervals_free_space"))
        if np.array_equal(pp.spec, base.spec):
            pars.append(pp.par); xs.append(np.clip(pp.x0, pp.xl, pp.xu))
    return base.spec, np.stack(pars), np.stack(xs)


@pytest.mark.parametrize("name", ["corridors8_3d", "waypoints3d"])
def test_host_build_follows_scipy_core(native_lib, hostsim, name):
    """The source the kernels are compiled from is right at this size: the single-lane host build and scipy's compiled
    SLSQP core, fed the same evaluations, take the same iterations to the same point."""
    pp = _packed(name)
    assert pp.layout.n > 100
    ref = hostsim_loader.scipy_core_solve(hostsim, pp, maxiter=500)
    mine = hostsim.solve(pp, maxiter=500)
    assert (mine["status"], mine["nit"]) == (ref["status"], ref["nit"]) == (0, ref["nit"])
    assert np.abs(mine["x"] - ref["x"]).max() <= 1e-5


@pytest.mark.gpu
def test_plan_places_scratch_in_global_memory_only_where_it_does_not_fit(native_lib, monkeypatch):
    from trajectory_generator_b200 import batch, synthetic as syn
    for k in ("TG_QP_FAR", "TG_LS_FAR", "TG_QP_GS", "TG_LS_GS", "TG_QP_STAGED"):
        monkeypatch.delenv(k, raising=False)
    want = dict(corridors8_3d=(1, 0), waypoints3d=(1, 0), extreme3d=(1, 1))
    for name, (qp, ls) in want.items():
        plan = batch.solve_plan(_packed(name).spec, 4096)
        assert (plan["qp_far"], plan["ls_far"]) == (qp, ls), (name, plan)
        assert plan["gs_qp"] == 64 and plan["staged"] == 0 and plan["slots"] > 0
    for name in problems.ALL:
        plan = batch.solve_plan(_packed(name, problems.ALL[name]).spec, 4096)
        assert (plan["qp_far"], plan["ls_far"], plan["slots"], plan["slot_kib"]) == (0, 0, 0, 0), (name, plan)
    for name in syn.CONFIGS:
        plan = batch.solve_plan(syn.make(name, 4).spec, 65536)
        assert (plan["qp_far"], plan["ls_far"], plan["slots"]) == (0, 0, 0), (name, plan)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["fd", "analytic"])
@pytest.mark.parametrize("name", list(LARGE))
def test_solve_matches_hostsim(native_lib, hostsim, name, mode):
    """As tests/test_gpu_first.py::test_solve_matches_hostsim, at the far side of the placement rule.  In fd mode the
    forward differences (steps of 1.5e-8) magnify the last-bit differences of the lane folds by ~1e8, so on a problem
    with several local minima the two builds may settle in different ones (waypoints3d: 174 against 145 iterations,
    f 0.43184 against 0.43327, measured on a B200): there the device solve must converge to a point no worse than the
    host build's."""
    from trajectory_generator_b200 import batch
    pp = _packed(name)
    L = pp.layout
    ref = hostsim.solve(pp, maxiter=MAXITER[name], fd=mode == "fd")
    out = batch.solve_host(pp.spec, pp.par[None], np.clip(pp.x0, pp.xl, pp.xu)[None], maxiter=MAXITER[name], jacobian=mode)
    dcp = np.abs(out["x"][0][:L.ia + 1] - ref["x"][:L.ia + 1]).max()
    print(name, mode, "gpu", int(out["status"][0]), int(out["nit"][0]), "host", ref["status"], ref["nit"], dcp)
    if ref["status"] == 0:
        assert int(out["status"][0]) == 0
        tol = 1e-5 * max(1.0, abs(ref["f"]))
        if mode == "fd" and float(out["f"][0]) < ref["f"] - tol:
            return
        assert abs(float(out["f"][0]) - ref["f"]) <= tol
        assert dcp <= 1e-3


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(LARGE))
def test_early_iterates_match_hostsim(native_lib, hostsim, name):
    """Cut off after 1, 2 and 5 iterations, the device iterate is the host build's up to the order of the lane folds."""
    from trajectory_generator_b200 import batch
    pp = _packed(name)
    for maxiter in (1, 2, 5):
        ref = hostsim.solve(pp, maxiter=maxiter)
        out = batch.solve_host(pp.spec, pp.par[None], np.clip(pp.x0, pp.xl, pp.xu)[None], maxiter=maxiter)
        err = np.abs(out["x"][0] - ref["x"]).max() / np.abs(ref["x"]).max()
        print(name, maxiter, "relative difference %.2e" % err)
        assert int(out["status"][0]) == ref["status"] == 9
        assert err <= 1e-8, (name, maxiter, err)


def _same(a, b):
    for k in ("x", "status", "nit", "f", "violation"):
        assert np.array_equal(a[k], b[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("switch,lanes", [("TG_QP_FAR", ("TG_QP_GS", "64")), ("TG_LS_FAR", ("TG_LS_GS", "32"))])
def test_forced_global_placement_is_bit_identical(native_lib, monkeypatch, switch, lanes):
    """TG_QP_FAR=1 / TG_LS_FAR=1 move a stage's scratch of shapes that fit to workspace slots; the far kernels run with 64
    (QP) / 32 (line search) lanes, so the reference run pins the same lane count: only the addresses differ."""
    from trajectory_generator_b200 import batch, synthetic as syn
    monkeypatch.setenv(*lanes)
    for name in ("C2", "C4"):
        b = syn.make(name, 512)
        for mode in ("fd", "analytic"):
            monkeypatch.delenv(switch, raising=False)
            assert batch.solve_plan(b.spec, 512)[switch.lower()[3:]] == 0
            ref = batch.solve_host(b.spec, b.par, b.x0, jacobian=mode)
            monkeypatch.setenv(switch, "1")
            plan = batch.solve_plan(b.spec, 512)
            assert plan[switch.lower()[3:]] == 1 and plan["slots"] > 0
            _same(batch.solve_host(b.spec, b.par, b.x0, jacobian=mode), ref)


@pytest.mark.gpu
@pytest.mark.parametrize("slices", [None, "2"])
def test_slots_do_not_alias(native_lib, monkeypatch, slices):
    """One problem gives the same bits alone and at any position of a batch whose lane groups reuse their slots."""
    from trajectory_generator_b200 import batch
    if slices:
        monkeypatch.setenv("TG_SLICES", slices)
    spec, par, x0 = _perturbed("corridors8_3d", 2048, seed=5)
    alone = batch.solve_host(spec, par[:1], x0[:1], jacobian="fd")
    for pos in (0, 1, 777, 2047):
        p, x = par.copy(), x0.copy()
        p[pos], x[pos] = par[0], x0[0]
        out = batch.solve_host(spec, p, x, jacobian="fd")
        for k in ("x", "status", "nit", "f", "violation"):
            assert np.array_equal(out[k][pos], alone[k][0]), (pos, k)


@pytest.mark.gpu
def test_generate_trajectories_mixes_large_and_small_shapes(native_lib):
    from trajectory_generator_b200.trajectory_generator import TrajectoryGenerator
    ns = helpers.product_namespace()
    items = [problems.sfc3d_four(ns), corridors8_3d(ns), problems.sfc3d_four(ns), waypoints3d(ns), corridors8_3d(ns)]
    gen = TrajectoryGenerator(3, maxiter=500)
    kw = items[3][2]          # (the corridor problems take their intervals from the corridors)
    many = gen.generate_trajectories([it[1] for it in items], **kw)
    assert len(many) == len(items)
    for it, res in zip(items, many):
        one = gen.generate_trajectory(it[1], **kw)
        assert res.control_points.shape == one[0].shape
        assert np.array_equal(res.control_points, one[0]) and res.scale_factor == one[1]


@pytest.mark.gpu
def test_dropin_generate_trajectory_on_a_long_corridor_path(native_lib):
    from trajectory_generation.trajectory_generator import TrajectoryGenerator
    d, cc, kw = corridors8_3d(helpers.product_namespace())
    gen = TrajectoryGenerator(3, maxiter=500)
    cps, scale, viol = gen.generate_trajectory(cc, **kw)
    assert cps.shape == (3, 49) and cps.dtype == np.float64
    r = gen.last_result
    assert r.status == 0 and not viol
    assert np.array_equal(cps.flatten(), r.x[:cps.size]) and scale == r.x[cps.size]


@pytest.mark.gpu
def test_corridor_problems_of_a_long_path(native_lib):
    import torch
    from trajectory_generator_b200.batched import CorridorProblems
    rng = np.random.default_rng(3)
    B = 256
    pts = np.repeat(np.concatenate(PTS8, 1)[None], B, 0)
    pts[:, :, 1:-1] += rng.uniform(-0.3, 0.3, (B, 3, 7))
    pads = np.tile(np.array([2.5, 2.4, 2.8]), (B, 8, 1))
    v0 = pts[:, :, 1] - pts[:, :, 0]; v0 /= np.linalg.norm(v0, 2, 1)[:, None]
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    cp = CorridorProblems(3, corridor_points=t(pts), corridor_pads=t(pads), min_intervals_per_corridor=2,
                          start_velocity=t(v0), end_zero_velocity=True, max_velocity=5.0, max_acceleration=0.3,
                          objective_function_type="minimal_velocity_path")
    assert max(sum(ipc) for ipc, _ in cp.shapes()) >= 46
    out = cp.solve(maxiter=500)
    assert (out["status"] == 0).double().mean().item() > 0.8


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(LARGE))
def test_workspace_of_exactly_the_reported_size(native_lib, hostsim, name):
    """tg_solve_workspace_bytes counts the slots: a solve with buffers of exactly that size runs, and the evaluation
    kernel runs at this size too (values against the host build)."""
    import torch
    from trajectory_generator_b200 import batch
    spec, par, x0 = _perturbed(name, 64, seed=9) if name != "extreme3d" else (lambda p: (p.spec, p.par[None].repeat(64, 0), np.clip(p.x0, p.xl, p.xu)[None].repeat(64, 0)))(_packed(name))
    bufs = batch.SolveBuffers(spec, 64, torch.device("cuda:0"))
    assert bufs.ws.numel() == native_lib.tg_solve_workspace_bytes(bufs.sp, 64) > 0
    out = batch.solve(spec, torch.from_numpy(par).cuda(), torch.from_numpy(x0).cuda(), maxiter=3, buffers=bufs)
    assert (out["status"] == 9).all()
    pp = _packed(name)
    f, g, c, _ = hostsim.eval(pp, np.clip(pp.x0, pp.xl, pp.xu))
    ev = batch.evaluate_host(pp.spec, pp.par[None], np.clip(pp.x0, pp.xl, pp.xu)[None], want=("f", "g", "c"))
    assert helpers.relerr(ev["c"][0], c) <= 1e-12 and abs(ev["f"][0] - f) <= 1e-12 * max(1.0, abs(f))
