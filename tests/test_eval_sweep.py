"""The evaluation kernels against the oracle over a seeded sweep of shapes: 2-D and 3-D, every objective, every turning
kind, tangential bounds, intermediate waypoints, obstacles and 1-8 uneven corridors, with interval counts on both sides
of every lane-pass edge of the 8 / 16 / 32-lane groups (a lane-strided loop over intervals or items takes several passes
from 33 intervals on) up to 509 intervals (N = 512 control points, the largest shape the library accepts).

The fixtures of tests/problems.py have at most 30 intervals, so there every lane-strided loop runs one pass.  Here the
per-lane running best, the fold that carries the arg index (tg_wargmax / tg_wargmin) and the rule that the winning lane
writes the gradient run over several passes, at every lane-group size (TG_EVAL_GS), on the constraint-value sink of
calls without `c`, and for long shapes whose lane groups do not all fit in one CTA's shared memory."""
import numpy as np
import pytest

import helpers
import problems

OBJECTIVES = ("minimal_time_path", "minimal_distance_path", "minimal_velocity_path", "minimal_acceleration_path",
              "minimal_distance_and_time_path", "minimal_velocity_and_time_path", "minimal_acceleration_and_time_path",
              "minimal_time_path_velocity_penalty")
TURNING = ("curvature", "angular_rate", "centripetal_acceleration")
GROUP_SIZES = (8, 16, 32)
# intervals of the free-space cases (509 twice: once in 2-D, once in 3-D)
NINT = (5, 8, 9, 16, 17, 31, 32, 33, 64, 65, 130, 509, 509)
# obstacle counts of the free-space cases: K * nint lands on or next to a multiple of 32 (16 * 2, 17 * 2, 31 * 1,
# 33 * 1, 9 * 7, 65 * 1 ...); 0 = none
OBSTACLES = (3, 4, 7, 2, 2, 1, 0, 1, 1, 1, 0, 2, 3)
# corridor cases: (dimension, intervals per corridor, obstacles inside the corridors)
CORRIDORS = ((2, (9,), 0), (3, (5, 7, 5), 2), (2, (9, 7, 8, 9), 0), (3, (13, 14, 12, 13, 13), 1),
             (2, (20, 25, 21, 22, 20, 22), 3), (3, (15,) * 8, 0), (3, (63,) * 8, 2))
JAC_ALL_COLUMNS = 200          # up to this many variables every Jacobian column is checked


def _free_case(ns, k, nint, n_obs):
    """Seeded random container in free space (the field mix of tests/test_packing.py's random containers), with the
    objective, the turning kind and the dimension cycled by case number so that the sweep covers each of them."""
    W, WD, DB, TB, Ob, CC = (ns[q] for q in ("Waypoint", "WaypointData", "DerivativeBounds", "TurningBound", "Obstacle",
                                              "ConstraintsContainer"))
    rng = np.random.default_rng(20261020 + k)
    d = 2 + k % 2
    vec = lambda s=3.0: rng.normal(size=(d, 1)) * s
    start, end = vec(), vec() + 8.0

    def terminal(loc):
        kind = rng.integers(0, 4)
        kw = dict(location=loc)
        if kind == 0:
            kw["velocity"] = vec(1.0)
        elif kind == 1:
            kw["velocity"] = np.zeros((d, 1))
        elif kind == 2:
            kw["velocity"] = np.zeros((d, 1)); kw["direction"] = vec(1.0)
        else:
            kw["velocity"] = vec(1.0); kw["acceleration"] = vec(0.5)
        return W(**kw)
    wps = [terminal(start)]
    niw = 2 if k % 3 == 2 else int(rng.integers(0, 2))
    with_iv = rng.random() < 0.5
    for i in range(niw):
        wps.append(W(location=start + (end - start) * (i + 1) / (niw + 1) + vec(0.5), velocity=vec(1.0) if with_iv else None))
    wps.append(terminal(end))
    f = dict(max_velocity=float(rng.uniform(3, 9)))
    if rng.random() < 0.6: f["max_acceleration"] = float(rng.uniform(1, 9))
    if rng.random() < 0.4: f["max_jerk"] = float(rng.uniform(1, 9))
    if rng.random() < 0.3: f["gravity"] = float(rng.uniform(0.1, 1))
    if rng.random() < 0.4: f["min_velocity"] = float(rng.uniform(0.01, 0.5))
    if rng.random() < 0.4: f["max_upward_velocity"] = f["max_velocity"] * 0.5
    if rng.random() < 0.4: f["max_horizontal_velocity"] = f["max_velocity"] * 0.8
    if k % 4 == 1:
        f["min_tangential_acceleration"] = -float(rng.uniform(1, 5)); f["max_tangential_acceleration"] = float(rng.uniform(1, 5))
    tb = TB(float(rng.uniform(0.5, 5)), TURNING[k % 3])
    obs = [Ob(center=start + (end - start) * rng.random() + vec(0.5), radius=float(rng.uniform(0.2, 1)))
           for _ in range(n_obs)] or None
    cc = CC(WD(tuple(wps)), DB(**f), tb, None, obs)
    return d, cc, dict(objective_function_type=OBJECTIVES[k % len(OBJECTIVES)], num_intervals_free_space=nint)


def _corridor_case(ns, k, d, ipc, n_obs):
    """Seeded corridor path with the given (uneven) intervals per corridor, as tests/problems.py:sfc_obstacles3d with
    obstacles inside the corridors when n_obs > 0."""
    W, WD, DB, TB, Ob = ns["Waypoint"], ns["WaypointData"], ns["DerivativeBounds"], ns["TurningBound"], ns["Obstacle"]
    rng = np.random.default_rng(777 + k)
    pts = [np.zeros((d, 1))]
    for _ in ipc:
        step = rng.uniform(-1, 1, (d, 1)); step[0, 0] = 0
        pts.append(pts[-1] + step * 3 + np.eye(d)[:, :1] * rng.uniform(4, 7))
    rot = ns["get%dDRotationAndTranslationFromPoints" % d]
    sfcs = []
    for i in range(len(ipc)):
        R, T, L = rot(pts[i], pts[i + 1])
        sfcs.append(ns["SFC"](np.array([[L + 2.5]] + [[rng.uniform(2, 3)]] * (d - 1)), T, R))
    sfc = ns["SFC_Data"](tuple(sfcs), np.concatenate(pts, 1), 1, intervals_per_corridor=np.array(ipc))
    v0 = (pts[1] - pts[0]) / np.linalg.norm(pts[1] - pts[0])
    wd = WD((W(location=pts[0], velocity=v0), W(location=pts[-1], velocity=np.zeros((d, 1)))))
    tb = TB(float(rng.uniform(1, 4)), TURNING[k % 3]) if k % 2 else None
    cc = ns["ConstraintsContainer"](waypoint_constraints=wd, derivative_constraints=DB(5, 0.3 + rng.random()),
                                    turning_constraint=tb, sfc_constraints=sfc)
    if n_obs:
        cc.obstacle_constraints = [Ob(center=(pts[i] + pts[i + 1]) / 2 + rng.uniform(-0.3, 0.3, (d, 1)), radius=0.4)
                                   for i in range(n_obs)]
    return d, cc, dict(objective_function_type=OBJECTIVES[(k + 3) % len(OBJECTIVES)])


def _case_names():
    return ["free%d_%dd_nint%d_obs%d" % (k, 2 + k % 2, nint, K) for k, (nint, K) in enumerate(zip(NINT, OBSTACLES))] + \
           ["sfc%d_%dd_%dx%s_obs%d" % (k, d, len(ipc), "-".join(map(str, sorted(set(ipc)))), K)
            for k, (d, ipc, K) in enumerate(CORRIDORS)]


CASES = _case_names()


def _case(name):
    """(pack_problem result, oracle) of a sweep case by name."""
    import tg_oracle
    from trajectory_generator_b200.problem import pack_problem
    ns = helpers.product_namespace()
    k = int(name.split("_")[0][3 if name.startswith("sfc") else 4:])
    if name.startswith("free"):
        d, cc, kw = _free_case(ns, k, NINT[k], OBSTACLES[k])
    else:
        d, cc, kw = _corridor_case(ns, k, *CORRIDORS[k])
    obj = kw["objective_function_type"]
    pp = pack_problem(d, cc, obj, kw.get("num_intervals_free_space"))
    op = tg_oracle.OracleProblem(d, cc, obj, kw.get("num_intervals_free_space"))
    return pp, op


def _points(pp, seeds=(1, 2)):
    L = pp.layout
    return np.stack([np.clip(problems.test_point(pp.x0, L.d, L.N, s), pp.xl, pp.xu) for s in seeds])


def _tie_point(pp):
    """Control points repeating every 4 indices (a lopsided closed loop traced over and over; small exact binary values,
    so intervals 4 apart give bit-identical values on every build, while the 4 intervals of one period differ by far
    more than rounding): every max / min over intervals or hull points is tied across lanes, and the reference's upward
    scan with a strict comparison makes the lowest index the winner."""
    L = pp.layout
    x = _points(pp, (3,))[0]
    loop = np.array([[0, 1, 1.5, 0.25], [0, 0.25, 1, 0.75], [0, 0.5, 0.75, 0.25]])
    for c in range(L.d):
        x[c * L.N:(c + 1) * L.N] = loop[c][np.arange(L.N) % 4]
    x[L.ia] = 1.0
    return x


def _is_linear(L, r):
    return r < L.r_sder or (L.r_sfcl <= r < L.r_obs)


def _nonlinear_rows(L):
    return np.array([r for r in range(L.m) if not _is_linear(L, r)], dtype=int)


def _columns(pp, x, jacs, gs_list=GROUP_SIZES):
    """Jacobian columns to check: all of them up to JAC_ALL_COLUMNS variables; beyond, a seeded sample of 16 plus the
    alpha column, the control points of the first and last interval, one control point of every interval at a
    lane-pass edge (j = GS - 1, GS, 2 GS - 1, 2 GS, ...) and every column the max / min rows (all nonlinear rows but the
    per-interval tangential ones) touch in any of the given Jacobians [.., m_nl, n] -- the winning intervals."""
    L = pp.layout
    if L.n <= JAC_ALL_COLUMNS:
        return None
    cols = {L.ia}
    for c in range(L.d):
        cols.update(range(c * L.N, c * L.N + 4))
        cols.update(range((c + 1) * L.N - 4, (c + 1) * L.N))
    for gs in gs_list:
        for j in range(gs - 1, L.nint, gs):
            for jj in (j, j + 1):
                if jj < L.nint:
                    cols.add((jj % L.d) * L.N + jj + jj % 4)
    nl = _nonlinear_rows(L)
    keep = np.array([not (L.r_tanl <= r < L.r_tanl + L.n_tan // 2 or L.r_tanu <= r < L.r_tanu + L.n_tan // 2)
                     for r in nl], dtype=bool)
    for J in jacs:
        J = np.asarray(J).reshape(-1, len(nl), L.n)[:, keep]
        cols.update(np.nonzero(np.any(J != 0, axis=(0, 1)))[0].tolist())
    cols.update(np.random.default_rng(L.n).choice(L.n, 16, replace=False).tolist())
    return np.array(sorted(cols))


def _check_against_oracle(pp, op, x, f, g, c, jnl, cols, what):
    """Values to 1e-12 relative; gradient and nonlinear Jacobian rows to 1e-9 on the entries the central-difference
    oracle vouches for (>= 97 % of them).  g [k, n] and jnl [k, m_nl, n] hold k evaluations of the same point (one per
    lane-group size): the oracle runs once for all of them."""
    L = pp.layout
    fo = op.fun(x)
    assert np.all(np.abs(np.asarray(f) - fo) <= 1e-12 * max(1.0, abs(fo))), (what, f, fo)
    co = op.cons(x)
    for ck in np.atleast_2d(c):
        assert helpers.relerr(ck, co) <= 1e-12, (what, helpers.relerr(ck, co))
    nl = _nonlinear_rows(L)
    # (the objective of a long trajectory sums thousands of terms: its differences are taken in extended precision, or
    # the rounding of f over the stencil's step leaves the oracle unable to vouch for its entries)
    checks = [("g", np.asarray(g)[..., None, :], lambda z: np.atleast_1d(op.fun(np.asarray(z, dtype=np.longdouble))))]
    if len(nl):
        checks.append(("jnl", np.asarray(jnl), lambda z: op.cons(z)[nl]))
    for key, J, fun in checks:
        e, trusted = op.jacobian_error(J, x, fun=fun, cols=cols)
        assert trusted.mean() >= 0.97, (what, key, trusted.mean())
        assert np.all(e[..., trusted] <= 1e-9), (what, key, np.max(e[..., trusted]))


def _evaluate(pp, xs, monkeypatch, gs, want=("f", "g", "c", "jnl")):
    import torch
    from trajectory_generator_b200 import batch
    monkeypatch.setenv("TG_EVAL_GS", str(gs))
    dev = torch.device("cuda:0")
    par = torch.tensor(np.repeat(pp.par[None], len(xs), 0), device=dev)
    out = batch.evaluate(pp.spec, par, torch.tensor(xs, device=dev), want=want)
    return {k: v.cpu().numpy() for k, v in out.items()}


def test_sweep_covers_what_it_claims(native_lib):
    """The generator builds the shapes the sweep is about (host only: packing and the oracle's row count)."""
    seen = dict(d=set(), obj=set(), turn=set(), nint=set(), tan=0, iw=0, ncorr=set(), kn=set())
    for name in CASES:
        pp, op = _case(name)
        L = pp.layout
        assert (L.n, L.m, L.meq) == (op.n, op.m, op.meq), name
        seen["d"].add(L.d); seen["obj"].add(op.objective); seen["nint"].add(L.nint)
        seen["turn"].add(op.tb.bound_type if op.tb is not None else None)
        seen["tan"] += L.n_tan > 0; seen["iw"] += L.niw > 0
        seen["ncorr"].add(len(op.sfc.get_sfc_list()) if op.sfc is not None else 0)
        seen["kn"].add(L.n_obs * L.nint)
    assert seen["d"] == {2, 3} and seen["obj"] == set(OBJECTIVES) and set(TURNING) <= seen["turn"]
    assert set(NINT) <= seen["nint"] and {120, 504} <= seen["nint"] and seen["tan"] >= 2 and seen["iw"] >= 3
    assert {0, 1, 3, 4, 5, 6, 8} <= seen["ncorr"]
    assert {31, 32, 33, 34} <= seen["kn"] and max(seen["kn"]) > 32 * 8


@pytest.mark.parametrize("name", ["free10_2d_nint130_obs0", "free11_3d_nint509_obs2", "free12_2d_nint509_obs3"])
def test_host_build_matches_the_oracle_on_long_shapes(native_lib, hostsim, name):
    """The single-lane host build of the kernel source against the oracle at N = 133 and N = 512: values, linear rows,
    gradient and nonlinear Jacobian rows.  A device failure on these shapes is then a matter of lanes or launches."""
    pp, op = _case(name)
    L = pp.layout
    lin = op.linear_jacobian()
    rows = ~np.isnan(lin[:, 0])
    nl = _nonlinear_rows(L)
    for x in _points(pp):
        f, g, c, J = hostsim.eval(pp, x)
        assert np.abs(J[rows] - lin[rows]).max() <= 1e-15 if rows.any() else True
        _check_against_oracle(pp, op, x, f, g, c, J[nl], _columns(pp, x, [J[nl]]), name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_evaluation_matches_the_oracle_at_every_group_size(native_lib, hostsim, monkeypatch, name):
    """At 8, 16 and 32 lanes per problem: f, c to 1e-12 and g, jnl to 1e-9 of the oracle at two points; the call
    without `c` (constraint rows in the shared-memory sink) returns bit for bit what the full call returns; and at a
    point where every max / min is tied across lanes, the device picks the reference's winner (the lowest index) --
    the same rows as the single-lane host build."""
    pp, op = _case(name)
    L = pp.layout
    xs = _points(pp)
    xt = _tie_point(pp)
    outs = {}
    for gs in GROUP_SIZES:
        full = _evaluate(pp, np.concatenate([xs, xt[None]]), monkeypatch, gs)
        sink = _evaluate(pp, np.concatenate([xs, xt[None]]), monkeypatch, gs, want=("f", "g", "jnl"))
        for k in ("f", "g", "jnl"):
            assert np.array_equal(sink[k], full[k]), (name, gs, k)
        outs[gs] = full
    hf, hg, hc, hJ = hostsim.eval(pp, xt)
    for gs, o in outs.items():
        assert helpers.relerr(o["f"][2], hf) <= 1e-12 and helpers.relerr(o["c"][2], hc) <= 1e-12, (name, gs)
        assert helpers.relerr(o["g"][2], hg) <= 1e-12, (name, gs)
        assert helpers.relerr(o["jnl"][2], hJ[_nonlinear_rows(L)]) <= 1e-12, (name, gs, "tie point")
    for p, x in enumerate(xs):
        jnl = np.stack([outs[gs]["jnl"][p] for gs in GROUP_SIZES])
        _check_against_oracle(pp, op, x, [outs[gs]["f"][p] for gs in GROUP_SIZES],
                              np.stack([outs[gs]["g"][p] for gs in GROUP_SIZES]),
                              np.stack([outs[gs]["c"][p] for gs in GROUP_SIZES]), jnl,
                              _columns(pp, x, [jnl, hostsim.eval(pp, x)[3][_nonlinear_rows(L)]]), (name, p))


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_linear_rows_equal_the_oracle(native_lib, name):
    """batch.linear_rows (tg_linear_rows_batch): the constant rows of the linear blocks equal the oracle's to 1e-15,
    the nonlinear rows are zero."""
    import torch
    from trajectory_generator_b200 import batch
    pp, op = _case(name)
    A = batch.linear_rows(pp.spec, torch.tensor(np.stack([pp.par] * 3), device="cuda:0")).cpu().numpy()
    lin = op.linear_jacobian()
    rows = ~np.isnan(lin[:, 0])
    assert rows.any()
    for a in A:
        assert np.abs(a[rows] - lin[rows]).max() <= 1e-15, name
        assert not a[~rows].any(), name


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["free11_3d_nint509_obs2", "sfc6_3d_8x63_obs2"])
@pytest.mark.parametrize("want", [("f", "g", "c", "jnl"), ("f", "g", "jnl")])
def test_ragged_batches_of_long_shapes(native_lib, monkeypatch, name, want):
    """Rows of a ragged batch (1, 3, 33 problems at an offset) are bit for bit those of the full batch, with lane groups
    that take several passes and CTAs that hold fewer lane groups than 128 / GS."""
    pp, _ = _case(name)
    L = pp.layout
    xs = _points(pp, range(100, 180))
    for gs in GROUP_SIZES:
        full = _evaluate(pp, xs, monkeypatch, gs, want)
        for lo, cnt in ((0, 1), (5, 3), (40, 33)):
            part = _evaluate(pp, xs[lo:lo + cnt], monkeypatch, gs, want)
            for k in want:
                assert np.array_equal(part[k], full[k][lo:lo + cnt]), (name, gs, k, lo, cnt)


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", ["C2", "C3", "C4", "C5a", "C5c"])
def test_fixed_shape_and_generic_evaluation(native_lib, monkeypatch, cfg):
    """The benchmark's configurations run kernels instantiated for their fixed shape (tg_shape.h); TG_GENERIC_KERNELS=1
    runs the generic ones.  Both meet the oracle.  Against each other: the objective and its gradient are bit-identical,
    and so is all of C4; elsewhere the constraint rows and their Jacobian differ in the last places, where the compiler
    contracts the folded constant-descriptor arithmetic into FMAs differently (measured on a B200: c up to 3.6e-14,
    jnl up to 9.8e-13 relative, both C3)."""
    import torch
    import tg_oracle
    from trajectory_generator_b200 import batch, synthetic as syn
    from trajectory_generator_b200.problem import pack_problem
    b = syn.make(cfg, 64)
    xe = syn.evaluation_points(b)
    dev = torch.device("cuda:0")

    def run():
        out = batch.evaluate(b.spec, torch.tensor(b.par, device=dev), torch.tensor(xe, device=dev))
        return {k: v.cpu().numpy() for k, v in out.items()}
    monkeypatch.delenv("TG_GENERIC_KERNELS", raising=False)
    fixed = run()
    monkeypatch.setenv("TG_GENERIC_KERNELS", "1")
    generic = run()
    for i in (0, 1, 2, 63):
        d, cc, kw = syn.container_for(b, i)
        obj = kw.get("objective_function_type", syn.OBJECTIVE[cfg])
        op = tg_oracle.OracleProblem(d, cc, obj, kw.get("num_intervals_free_space"))
        assert np.array_equal(pack_problem(d, cc, obj, kw.get("num_intervals_free_space")).spec, b.spec)
        for o in (fixed, generic):
            _check_against_oracle(b, op, xe[i], o["f"][i], o["g"][i], o["c"][i], o["jnl"][i], None, (cfg, i))
    print(cfg, "bit-identical", {k: bool(np.array_equal(fixed[k], generic[k])) for k in fixed},
          "relative difference", {k: helpers.relerr(fixed[k], generic[k]) for k in fixed})
    for k in ("f", "g") + (("c", "jnl") if cfg == "C4" else ()):
        assert np.array_equal(fixed[k], generic[k]), (cfg, k)
    assert helpers.relerr(fixed["c"], generic["c"]) <= 1e-13, cfg
    assert helpers.relerr(fixed["jnl"], generic["jnl"]) <= 1e-11, cfg


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", ["C2", "C3", "C4"])
def test_fixed_shape_and_generic_solves_agree(native_lib, monkeypatch, cfg):
    """The benchmark's fixed-shape solve against the generic kernels (which the reference fixtures anchor), fd mode, 256
    problems, under the contract of tests/test_gpu_first.py::test_fused_and_lockstep_kernels_agree; C4, whose
    evaluations are bit-identical, solves bit for bit alike.  (C5a / C5c are left out: the reference itself lands
    elsewhere on most of them from x0 + 1 ulp (DESIGN.md section 5), and the last-place differences of the evaluation
    part the two runs in the same way -- measured on a B200: same status on 74 % of C5a, equal iteration counts on
    under 5 %.)"""
    from trajectory_generator_b200 import batch, synthetic as syn
    b = syn.make(cfg, 256)
    monkeypatch.delenv("TG_GENERIC_KERNELS", raising=False)
    a = batch.solve_host(b.spec, b.par, b.x0, jacobian="fd")
    monkeypatch.setenv("TG_GENERIC_KERNELS", "1")
    g = batch.solve_host(b.spec, b.par, b.x0, jacobian="fd")
    same = a["status"] == g["status"]
    ok = same & (a["status"] == 0) & (a["nit"] == g["nit"])
    print(cfg, "same status %.3f" % same.mean(), "converged with equal nit %.3f" % ok.mean(),
          "bit-identical x %.3f" % np.all(a["x"] == g["x"], 1).mean())
    assert same.mean() >= 0.9
    assert (np.abs(a["x"][ok] - g["x"][ok]).max(1) <= 1e-5).mean() >= 0.9
    if cfg == "C4":
        for k in ("x", "f", "status", "nit", "violation"):
            assert np.array_equal(a[k], g[k]), k
