"""Drop-in ``TrajectoryGenerator`` (reference TG/trajectory_generator.py:46-112) on the CUDA path.

``generate_trajectory`` keeps the reference signature and return value
``(control_points[d,N], scale_factor, is_violation)``; the SLSQP loop and everything it evaluates
run on the GPU (one warp per problem).  ``generate_trajectories`` is the batched addition: many
containers at once, grouped by problem shape; the groups are solved in one library call, concurrently on
the device (tg_solve_mixed_host).
"""
import numpy as np

from . import batch
from .constraint_data_structures.constraints_container import ConstraintsContainer
from .constraint_data_structures.waypoint_data import Waypoint
from .problem import PackedGroup, pack_problem, pack_problems


class TrajectoryResult:
    """Per-problem solver outcome that the reference keeps internal (OptimizeResult.status / nit / fun)."""

    def __init__(self, control_points, scale_factor, is_violation, status, nit, fun, x, start=0, max_violation=None,
                 multipliers=None, kkt=None, polish_status=None):
        """start: the multi-start start that won (0 without multi-start); max_violation: its true maximum constraint
        violation (computed by multi-start solves only, else None).  multipliers [m] / kkt [4]: the KKT multipliers of
        the last QP in constraint row order (scipy's OptimizeResult.multipliers; Layout.row_blocks names the rows) and
        the first-order optimality certificate (batch.KKT_FIELDS), with TrajectoryGenerator(..., multipliers=True)
        only, else None.  polish_status: the post-solve polish's code (batch.POLISH_STATUS) with
        TrajectoryGenerator(..., polish=True) only, else None."""
        self.control_points, self.scale_factor, self.is_violation = control_points, scale_factor, is_violation
        self.status, self.nit, self.fun, self.x = status, nit, fun, x
        self.start, self.max_violation = start, max_violation
        self.multipliers, self.kkt = multipliers, kkt
        self.polish_status = polish_status
        self.success = status == 0

    def __iter__(self):      # unpacks like the reference's return tuple
        return iter((self.control_points, self.scale_factor, self.is_violation))


class TrajectoryGenerator:
    def __init__(self, dimension: int, jacobian: str = "fd", maxiter: int = 100, ftol: float = 1e-6, starts: int = 1,
                 seed: int = 0, multipliers: bool = False, polish: bool = False):
        """jacobian: "fd" (default) forms derivatives on the GPU exactly as scipy does for the reference (2-point
        forward differences, h = 1.49e-8, bound-aware), so the iterates follow the reference's and the converged
        control points agree within 1e-5 wherever the reference reproduces itself to that level; "analytic" uses
        the closed-form Jacobians (1.3-1.8x faster; same optimum within what ftol resolves, different last digits).
        maxiter / ftol default to scipy's SLSQP defaults, which is what the reference runs with
        (TG/trajectory_generator.py:85).
        starts > 1: every problem is solved from `starts` seeded starts on the device (start 0 is the usual one) and the
        best converged feasible result is kept (batch.solve_mixed_multistart; DESIGN.md §4 *Multi-start*).
        multipliers: every TrajectoryResult also carries the KKT multipliers and the optimality certificate
        (DESIGN.md §4 *Multipliers and the KKT certificate*); the groups are then solved through the device entry
        points.
        polish: the converged problems are polished on the device after the solve (batch.polish; DESIGN.md §4 *Polish*):
        the results hold the polished x, and multipliers, kkt and polish_status are filled in (implies multipliers)."""
        if int(starts) < 1:
            raise ValueError("starts must be at least 1")
        self._dimension = dimension
        self._order = 3
        self._jacobian, self._maxiter, self._ftol = jacobian, maxiter, ftol
        self._starts, self._seed = int(starts), int(seed)
        self._polish = bool(polish)
        self._multipliers = bool(multipliers) or self._polish
        self.last_result = None

    # ---- reference API ---------------------------------------------------------------------------
    def generate_trajectory(self, constraints_container: ConstraintsContainer,
                            objective_function_type: str = "minimal_velocity_and_time_path",
                            num_intervals_free_space: int = None,
                            initial_control_points: np.ndarray = None,
                            initial_scale_factor: float = None):
        res = self.generate_trajectories([constraints_container], objective_function_type, num_intervals_free_space,
                                         [initial_control_points], [initial_scale_factor])[0]
        self.last_result = res
        return res.control_points, res.scale_factor, res.is_violation

    def get_terminal_waypoint_properties(self, control_points: np.ndarray, scale_factor: float, side: str):
        """TG/trajectory_generator.py:99-106 (CF/waypoint_constraints.py:149-203)."""
        P = np.asarray(control_points, dtype=float)
        a, b, c = (P[:, 0], P[:, 1], P[:, 2]) if side == "start" else (P[:, -3], P[:, -2], P[:, -1])
        if side not in ("start", "end"):
            raise Exception("Funtion does not support this side value")
        location = (a + 4 * b + c) / 6
        velocity = (c - a) / (2 * scale_factor)
        acceleration = (a - 2 * b + c) / (scale_factor * scale_factor)
        return Waypoint(location=location[:, None], velocity=velocity[:, None], acceleration=acceleration[:, None])

    # ---- batched addition ------------------------------------------------------------------------
    def generate_trajectories(self, containers, objective_function_type="minimal_velocity_and_time_path",
                              num_intervals_free_space=None, initial_control_points=None, initial_scale_factors=None):
        """Solves every container; problems of identical shape share one kernel launch.
        Returns a list of TrajectoryResult in input order.  Long lists go through in chunks of PIPELINE_CHUNK
        containers: a helper thread packs the next chunk while the GPU solves the current one (the library call
        releases the GIL), so the Python-side packing is hidden behind the solve or the other way round."""
        count = len(containers)
        results = [None] * count
        default_guess = initial_control_points is None and initial_scale_factors is None
        if default_guess and count > 2 * self.PIPELINE_CHUNK:
            from concurrent.futures import ThreadPoolExecutor
            bounds = list(range(0, count, self.PIPELINE_CHUNK)) + [count]
            pack = lambda a, b: pack_problems(self._dimension, containers[a:b], objective_function_type, num_intervals_free_space)
            with ThreadPoolExecutor(max_workers=1) as pool:
                pending = pool.submit(pack, bounds[0], bounds[1])
                for k in range(len(bounds) - 1):
                    groups = pending.result()
                    if k + 2 < len(bounds):
                        pending = pool.submit(pack, bounds[k + 1], bounds[k + 2])
                    self._solve_groups(groups, results, bounds[k])
            return results
        if default_guess:
            # vectorised packing: containers grouped by shape, one numpy gather per field (problem.pack_problems)
            self._solve_groups(pack_problems(self._dimension, containers, objective_function_type, num_intervals_free_space),
                               results, 0)
            return results
        icps = initial_control_points if initial_control_points is not None else [None] * count
        isfs = initial_scale_factors if initial_scale_factors is not None else [None] * count
        packed = [pack_problem(self._dimension, cc, objective_function_type, num_intervals_free_space, icps[i], isfs[i])
                  for i, cc in enumerate(containers)]
        by_key = {}
        for i, p in enumerate(packed):
            by_key.setdefault(p.key, []).append(i)
        groups = [PackedGroup(np.asarray(idx), packed[idx[0]].spec, np.stack([packed[i].par for i in idx]),
                              np.stack([np.clip(packed[i].x0, packed[i].xl, packed[i].xu) for i in idx]),
                              packed[idx[0]].xl, packed[idx[0]].xu) for idx in by_key.values()]
        self._solve_groups(groups, results, 0)
        return results

    # a solve has a fixed latency of ~100 lock-step rounds whatever its size (C2: ~50 ms), so chunks must be large for the
    # overlap to pay: lists of up to two chunks go through in one piece
    PIPELINE_CHUNK = 32768

    def _solve_groups(self, groups, results, offset):
        """one library call for the groups (shapes) of a chunk; results[offset + index] are filled in"""
        if self._starts > 1 or self._multipliers:
            return self._solve_groups_multistart(groups, results, offset)
        buckets = [(g.spec, g.par, g.x0) for g in groups]
        if len(buckets) == 1:
            outs = [batch.solve_host(*buckets[0], self._maxiter, self._ftol, self._jacobian)]
        else:       # different shapes: one call, the buckets' solves overlap on the device (tg_solve_mixed_host)
            outs = batch.solve_mixed_host(buckets, self._maxiter, self._ftol, self._jacobian)
        for g, out in zip(groups, outs):
            lay, idx = g.layout, g.indices
            xs = out["x"]
            cps_all = xs[:, :lay.d * lay.N].reshape(len(idx), lay.d, lay.N).copy()
            scales = xs[:, lay.ia].tolist(); viol = out["violation"].tolist(); status = out["status"].tolist()
            nit = out["nit"].tolist(); fs = out["f"].tolist()
            for k, i in enumerate(idx.tolist()):
                results[offset + i] = TrajectoryResult(cps_all[k], scales[k], bool(viol[k]), status[k], nit[k], fs[k], xs[k])
        return results

    def _solve_groups_multistart(self, groups, results, offset):
        """the groups moved to the current CUDA device and solved from self._starts starts each (one start: an ordinary
        device solve, batch.solve / solve_mixed)"""
        import torch
        dev = torch.device("cuda", torch.cuda.current_device())
        buckets = [(g.spec, torch.from_numpy(np.ascontiguousarray(g.par)).to(dev),
                    torch.from_numpy(np.ascontiguousarray(g.x0)).to(dev)) for g in groups]
        if self._starts > 1:
            outs = batch.solve_mixed_multistart(buckets, self._starts, self._seed, maxiter=self._maxiter, ftol=self._ftol,
                                                jacobian=self._jacobian, multipliers=self._multipliers,
                                                polish=self._polish)
        elif len(buckets) == 1:
            outs = [batch.solve(*buckets[0], maxiter=self._maxiter, ftol=self._ftol, jacobian=self._jacobian,
                                multipliers=True, polish=self._polish)]
        else:
            outs = batch.solve_mixed(buckets, self._maxiter, self._ftol, self._jacobian, multipliers=True,
                                     polish=self._polish)
        for g, out in zip(groups, outs):
            lay, idx = g.layout, g.indices
            out = {k: v.cpu().numpy() for k, v in out.items()}
            xs = out["x"]
            cps_all = xs[:, :lay.d * lay.N].reshape(len(idx), lay.d, lay.N).copy()
            for k, i in enumerate(idx.tolist()):
                results[offset + i] = TrajectoryResult(
                    cps_all[k], float(xs[k, lay.ia]), bool(out["violation"][k]), int(out["status"][k]), int(out["nit"][k]),
                    float(out["f"][k]), xs[k], int(out["best_start"][k]) if "best_start" in out else 0,
                    float(out["max_violation"][k]) if "max_violation" in out else None,
                    out["lam"][k] if self._multipliers else None, out["kkt"][k] if self._multipliers else None,
                    int(out["polish_status"][k]) if self._polish else None)
        return results
