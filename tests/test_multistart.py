"""Multi-start solves: K seeded starts per problem on the device, the best converged feasible one kept
(tg_multistart_expand / tg_multistart_select, batch.solve_multistart, TrajectoryGenerator(starts=...)).

The start model and the selection rule are restated here in numpy / plain Python; the device must reproduce the starts
bit for bit and pick the same winners."""
import math

import numpy as np
import pytest

import helpers
import problems

M64 = (1 << 64) - 1
KNOTS = 3
LADDER = (1.0, 0.5, 2.0, 0.75, 1.5, 0.625, 1.25, 3.0)


# ---------------------------------------------------------------------------------------------------------------------
# restatement of the start model (csrc/tg_multistart.cu)
# ---------------------------------------------------------------------------------------------------------------------
def splitmix64(z):
    z = (z + 0x9E3779B97F4A7C15) & M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def knot(seed, k, c, q):
    if q <= 0 or q > KNOTS:
        return 0.0
    h = splitmix64((splitmix64(seed & M64) + (k * 4 + c) * 8 + q) & M64)
    return float(h >> 11) * 2.0 ** -52 - 1.0


def profile(seed, k, c, j, N):
    W = N - 5
    t = (j - 2) * (KNOTS + 1)
    q = t // W
    w = (t % W) / W
    v0, v1 = knot(seed, k, c, q), knot(seed, k, c, q + 1)
    return v0 + w * (v1 - v0)


def expand(lay, par, x0, K, seed, spread):
    """(par_out [B*K, P], x_out [B*K, n]) of tg_multistart_expand"""
    d, N, ia = lay.d, lay.N, lay.ia
    par_out = np.repeat(par, K, axis=0)
    x_out = np.repeat(x0, K, axis=0)
    dl = [x0[:, c * N + N - 1] - x0[:, c * N] for c in range(d)]
    l2 = dl[0] * dl[0]
    for c in range(1, d):
        l2 = l2 + dl[c] * dl[c]
    scale = spread * np.sqrt(l2)
    for k in range(1, K):
        rows = x_out[k::K]
        rows[:, ia] = x0[:, ia] * LADDER[k % 8]
        for c in range(d):
            for j in range(3, N - 3):
                rows[:, c * N + j] = x0[:, c * N + j] + scale * profile(seed, k, c, j, N)
    return par_out, x_out


def max_violation(c, meq):
    """true maximum violation of constraint rows c [..., m] (NaN rows count as +inf)"""
    t = np.concatenate([np.abs(c[..., :meq]), np.maximum(0.0, -c[..., meq:])], -1)
    t = np.where(np.isnan(c), np.inf, t)
    return t.max(-1) if t.shape[-1] else np.zeros(c.shape[:-1])


def select(status, f, mv, tol):
    """winning start per problem: status [B, K], f [B, K], max violation [B, K]"""
    B, K = np.shape(status)
    out = np.zeros(B, dtype=np.int64)
    for b in range(B):
        best = None
        for k in range(K):
            ok = status[b][k] == 0 and mv[b][k] <= tol
            fk = math.inf if math.isnan(f[b][k]) else f[b][k]
            key = (0, fk, 0.0) if ok else (1, mv[b][k], fk)
            if best is None or key < best[0]:
                best = (key, k)
        out[b] = best[1]
    return out


def _batch(name, B):
    from trajectory_generator_b200 import synthetic
    return synthetic.make(name, B) if name != "large" else _large(B)


def _large(B):
    """the 8-corridor fixture of tests/test_large_shapes.py (N = 49, 3-D), B copies with shifted corridor points"""
    import test_large_shapes
    spec, par, x0 = test_large_shapes._perturbed("corridors8_3d", B, seed=5)

    class _B:
        pass
    b = _B()
    b.spec, b.par, b.x0 = spec, par, x0
    from trajectory_generator_b200.problem import Layout
    b.layout = Layout(spec)
    return b


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the restatements' properties
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["C2", "C4"])
def test_start_model_properties(native_lib, name):
    bt = _batch(name, 16)
    lay = bt.layout
    K = 8
    par_out, x_out = expand(lay, bt.par, bt.x0, K, seed=3, spread=0.1)
    assert np.array_equal(par_out, np.repeat(bt.par, K, axis=0))
    x = x_out.reshape(16, K, lay.n)
    assert np.array_equal(x[:, 0], bt.x0)                          # start 0 is the identity
    fixed = np.ones(lay.n, dtype=bool)
    for c in range(lay.d):
        fixed[c * lay.N + 3:c * lay.N + lay.N - 3] = False
    fixed[lay.ia] = False
    assert np.array_equal(x[:, :, fixed], np.repeat(bt.x0[:, None, fixed], K, 1))   # end points, scalars, times
    assert np.array_equal(x[:, :, lay.ia], bt.x0[:, None, lay.ia] * np.array(LADDER)[None, :K])
    assert all(np.any(x[:, k, ~fixed] != bt.x0[:, ~fixed]) for k in range(1, K))
    # no dependence on the batch position: a reversed batch gets the same starts per problem
    _, xr = expand(lay, bt.par[::-1].copy(), bt.x0[::-1].copy(), K, seed=3, spread=0.1)
    assert np.array_equal(xr.reshape(16, K, lay.n)[::-1], x)
    # another seed moves the interior points elsewhere, alpha the same way
    _, xs = expand(lay, bt.par, bt.x0, K, seed=4, spread=0.1)
    assert not np.array_equal(xs, x_out) and np.array_equal(xs.reshape(16, K, lay.n)[:, :, lay.ia], x[:, :, lay.ia])


def test_profile_and_knots():
    vals = [knot(s, k, c, q) for s in (0, 1, 2 ** 63) for k in range(1, 9) for c in range(3) for q in range(1, KNOTS + 1)]
    assert all(-1.0 <= v < 1.0 for v in vals) and len(set(vals)) == len(vals)
    assert knot(0, 1, 0, 0) == 0.0 and knot(0, 1, 0, KNOTS + 1) == 0.0
    for N in (7, 8, 11, 49):       # zero at the last fixed points j = 2 and j = N - 3, the knot values at the knots
        assert profile(9, 1, 0, 2, N) == 0.0 and profile(9, 1, 0, N - 3, N) == 0.0
    assert profile(9, 2, 1, 2 + 5, 25) == knot(9, 2, 1, 1)


def test_selection_rule():
    inf, nan = math.inf, math.nan
    tol = 1e-5
    cases = [
        # status, f, max violation -> winner
        (([0, 0, 0], [3.0, 2.0, 2.0], [0, 0, 0]), 1),                 # lowest f, tie -> lowest k
        (([9, 0, 0], [1.0, 5.0, 4.0], [0, 0, 1e-3]), 1),              # converged and feasible beats a lower f
        (([0, 9, 4], [1.0, 0.5, 0.1], [1e-3, 1e-4, 1e-4]), 2),        # none feasible: lowest violation, then lowest f
        (([9, 9], [2.0, 1.0], [0.5, 0.5]), 1),
        (([9, 8], [nan, 1.0], [0.5, 0.5]), 1),                        # NaN f ranks last
        (([0, 0], [1.0, 1.0], [inf, inf]), 0),                        # all infeasible, all tied
        (([0], [7.0], [0.0]), 0),
        (([0, 0], [2.0, nan], [0.0, 0.0]), 0),
        (([6, 0, 0], [1.0, 1.0, 1.0], [0.0, tol, tol * 1.01]), 1),    # the tolerance is inclusive
    ]
    for (status, f, mv), want in cases:
        assert select([status], [f], [mv], tol)[0] == want, (status, f, mv)
    c = np.array([[1e-3, -2e-3, 0.5, -0.25, nan], [0.0, 0.0, 1.0, 2.0, 3.0]])
    assert np.array_equal(max_violation(c[:, :4], 2), [0.25, 0.0])
    assert np.array_equal(max_violation(c, 2), [inf, 0.0])


def test_entry_points_fail_without_device(native_lib):
    """Without a device both entry points return an error and say why; bad arguments are named first."""
    import ctypes

    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    from trajectory_generator_b200 import _native, synthetic
    bt = synthetic.make("C2", 2)
    lay = bt.layout
    spec, sp = _native.spec_ptr(bt.spec)
    L = _native.lib()
    buf = np.zeros(64 * (lay.n + lay.P))
    p = ctypes.c_void_p(buf.ctypes.data)
    assert L.tg_multistart_expand(sp, 2, 0, p, p, 0, 0.1, p, p, None) != 0
    assert "at least 1" in L.tg_last_error().decode()
    assert L.tg_multistart_expand(sp, 2, 4, p, p, 0, 0.1, p, p, None) != 0
    assert "no CUDA device" in L.tg_last_error().decode()
    assert L.tg_multistart_select(sp, 2, 4, *([p] * 6), 1e-5, *([p] * 6), None, None) != 0
    assert "no CUDA device" in L.tg_last_error().decode()
    assert L.tg_multistart_select(sp, 2, 4, *([p] * 6), 1e-5, None, *([p] * 5), None, None) != 0
    assert "NULL" in L.tg_last_error().decode()
    from trajectory_generator_b200 import batch
    with pytest.raises(RuntimeError, match="CUDA tensors"):
        batch.solve_multistart(bt.spec, torch.from_numpy(bt.par), torch.from_numpy(bt.x0), 4)


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _np(out):
    return {k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in out.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("name,B", [("C2", 300), ("C4", 200), ("large", 6)])
@pytest.mark.parametrize("K,seed,spread", [(5, 0, 0.1), (9, 2 ** 64 - 1, 0.37)])
def test_expand_matches_restatement(native_lib, name, B, K, seed, spread):
    from trajectory_generator_b200 import batch
    bt = _batch(name, B)
    par_out, x_out = batch.multistart_expand(bt.spec, _dev(bt.par), _dev(bt.x0), K, seed, spread)
    want_par, want_x = expand(bt.layout, bt.par, bt.x0, K, seed, spread)
    assert np.array_equal(par_out.cpu().numpy(), want_par)
    assert np.array_equal(x_out.cpu().numpy().view(np.uint64), want_x.view(np.uint64))


def _same(a, b, keys=("x", "f", "status", "nit", "violation")):
    for k in keys:
        assert np.array_equal(np.asarray(a[k]).view(np.uint8), np.asarray(b[k]).view(np.uint8)), k


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["C2", "C4"])
@pytest.mark.parametrize("jacobian", ["analytic", "fd"])
def test_one_start_is_the_plain_solve(native_lib, name, jacobian):
    from trajectory_generator_b200 import batch
    bt = _batch(name, 256)
    x0 = _dev(bt.x0)
    ms = _np(batch.solve_multistart(bt.spec, _dev(bt.par), x0, 1, seed=11, jacobian=jacobian))
    assert np.array_equal(x0.cpu().numpy(), bt.x0)                  # the input is not overwritten
    ref = _np(batch.solve(bt.spec, _dev(bt.par), _dev(bt.x0), jacobian=jacobian))
    _same(ms, ref)
    assert np.all(ms["best_start"] == 0)


def _per_start(name, B, K, jacobian="analytic", seed=7):
    from trajectory_generator_b200 import batch
    bt = _batch(name, B)
    out = batch.solve_multistart(bt.spec, _dev(bt.par), _dev(bt.x0), K, seed=seed, jacobian=jacobian, return_all=True)
    return bt, _np(out), _np(out["all"])


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["C2", "C4"])
def test_per_start_results_are_plain_solves(native_lib, name):
    """start k's result is what batch.solve makes of the expanded row, in the batch and alone"""
    from trajectory_generator_b200 import batch
    K = 4
    bt, out, al = _per_start(name, 128, K)
    par_e, x_e = batch.multistart_expand(bt.spec, _dev(bt.par), _dev(bt.x0), K, 7)
    ref = _np(batch.solve(bt.spec, par_e, x_e.clone()))
    flat = {k: v.reshape((128 * K,) + v.shape[2:]) for k, v in al.items()}
    _same(flat, ref)
    for row in (0, 1, 5, 2 * K + 3, 127 * K + 2):
        one = _np(batch.solve(bt.spec, par_e[row:row + 1].clone(), x_e[row:row + 1].clone()))
        _same({k: v[row:row + 1] for k, v in flat.items()}, one)


@pytest.mark.gpu
@pytest.mark.parametrize("name,B", [("C2", 256), ("C4", 128), ("large", 4)])
def test_max_violation_and_winner(native_lib, name, B):
    """max_violation is the fold of batch.evaluate's rows; best_start is the restated rule on the per-start results"""
    import torch

    from trajectory_generator_b200 import batch
    K = 4
    bt, out, al = _per_start(name, B, K)
    lay = bt.layout
    xs = torch.from_numpy(al["x"].reshape(B * K, lay.n)).cuda()
    c = batch.evaluate(bt.spec, _dev(np.repeat(bt.par, K, axis=0)), xs, want=("c",))["c"].cpu().numpy()
    mv = max_violation(c, lay.meq).reshape(B, K)
    assert np.array_equal(al["max_violation"], mv)      # same instantiation, same lanes: the same bits
    want = select(al["status"], al["f"], mv, batch.MULTISTART_TOL)
    assert np.array_equal(out["best_start"], want)
    idx = np.arange(B)
    for k in ("x", "f", "status", "nit", "violation", "max_violation"):
        assert np.array_equal(out[k], al[k][idx, want]), k


@pytest.mark.gpu
def test_position_independence_and_determinism(native_lib):
    from trajectory_generator_b200 import batch
    bt = _batch("C2", 192)
    K = 4
    run = lambda par, x0: _np(batch.solve_multistart(bt.spec, _dev(par), _dev(x0), K, seed=5))
    base = run(bt.par, bt.x0)
    _same(run(bt.par, bt.x0), base, keys=("x", "f", "status", "nit", "violation", "best_start", "max_violation"))
    perm = np.random.default_rng(1).permutation(192)
    sh = run(bt.par[perm], bt.x0[perm])
    _same(sh, {k: v[perm] for k, v in base.items()}, keys=("x", "f", "status", "nit", "violation", "best_start", "max_violation"))
    for b in (0, 77):
        one = run(bt.par[b:b + 1], bt.x0[b:b + 1])
        _same(one, {k: v[b:b + 1] for k, v in base.items()}, keys=("x", "f", "status", "best_start", "max_violation"))


@pytest.mark.gpu
def test_pieces_match_one_piece(native_lib, monkeypatch):
    """a batch split into pieces under a small row cap gives the same bits as one piece"""
    from trajectory_generator_b200 import batch
    bt = _batch("C2", 100)
    args = (bt.spec, _dev(bt.par), _dev(bt.x0), 3)
    whole = _np(batch.solve_multistart(*args, seed=2))
    monkeypatch.setattr(batch, "MULTISTART_ROWS", 64)
    parts = _np(batch.solve_multistart(*args, seed=2))
    _same(parts, whole, keys=("x", "f", "status", "nit", "violation", "best_start", "max_violation"))


def _never_worse(s1, f1, ok1, s4, f4, ok4):
    assert np.sum(s4 == 0) >= np.sum(s1 == 0)
    assert np.all(ok4[ok1])
    assert np.all(f4[ok1] <= f1[ok1])


@pytest.mark.gpu
def test_never_worse_than_one_start(native_lib):
    from trajectory_generator_b200 import batch
    bt = _batch("C2", 1024)
    tol = batch.MULTISTART_TOL
    one = _np(batch.solve_multistart(bt.spec, _dev(bt.par), _dev(bt.x0), 1))
    four = _np(batch.solve_multistart(bt.spec, _dev(bt.par), _dev(bt.x0), 4))
    ok = lambda r: (r["status"] == 0) & (r["max_violation"] <= tol)
    _never_worse(one["status"], one["f"], ok(one), four["status"], four["f"], ok(four))


@pytest.mark.gpu
def test_drop_in_starts(native_lib):
    """TrajectoryGenerator(2, starts=4) over the 2-D golden solve fixtures, several shapes per call"""
    from trajectory_generator_b200 import batch
    from trajectory_generator_b200.problem import pack_problem
    from trajectory_generator_b200.trajectory_generator import TrajectoryGenerator
    ns = helpers.product_namespace()
    by_kw = {}
    for name in problems.SOLVE:
        d, cc, kw = problems.ALL[name](ns)
        if d == 2:
            by_kw.setdefault(tuple(sorted(kw.items())), []).append(cc)
    assert max(len(v) for v in by_kw.values()) >= 2
    for kw, ccs in by_kw.items():
        kw = dict(kw)
        ccs = ccs + ccs[:1]
        plain = TrajectoryGenerator(2).generate_trajectories(ccs, **kw)
        one = TrajectoryGenerator(2, starts=1).generate_trajectories(ccs, **kw)
        four = TrajectoryGenerator(2, starts=4, seed=3).generate_trajectories(ccs, **kw)
        for p, o in zip(plain, one):
            assert np.array_equal(p.x, o.x) and p.status == o.status and p.fun == o.fun and o.start == 0
        mv1 = []
        for cc, r in zip(ccs, one):      # the K = 1 results' true maximum violation, from the evaluation API
            pp = pack_problem(2, cc, kw.get("objective_function_type", "minimal_velocity_and_time_path"),
                              kw.get("num_intervals_free_space"))
            c = batch.evaluate_host(pp.spec, pp.par[None], r.x[None], want=("c",))["c"]
            mv1.append(max_violation(c, pp.layout.meq)[0])
        s1 = np.array([r.status for r in one]); f1 = np.array([r.fun for r in one])
        s4 = np.array([r.status for r in four]); f4 = np.array([r.fun for r in four])
        ok1 = (s1 == 0) & (np.array(mv1) <= batch.MULTISTART_TOL)
        ok4 = (s4 == 0) & (np.array([r.max_violation for r in four]) <= batch.MULTISTART_TOL)
        _never_worse(s1, f1, ok1, s4, f4, ok4)
        assert all(0 <= r.start < 4 for r in four)
        assert np.array_equal(four[0].x, four[-1].x)        # the same container twice: the same answer
