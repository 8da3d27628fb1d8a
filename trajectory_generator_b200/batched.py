"""Batched front end: B problems of one shape from arrays, assembled, solved and sampled on the GPU
(SURVEY.md 8(f) row f2: per-container packing in Python costs 170-400 us, 30-80x the GPU solve).

``BatchedProblem`` takes what a ``ConstraintsContainer`` holds, as CUDA tensors with a leading batch axis, and produces
the same (shape descriptor, parameter rows, initial variables) ``problem.pack_problem`` produces per container:

    bp = BatchedProblem(dimension=2, start=s, end=g, start_velocity=v0, end_velocity=v1,
                        max_velocity=2.0, max_acceleration=5.0, turning=("angular_rate", 1.8),
                        obstacle_centers=ctr, obstacle_radii=rad)
    out = bp.solve()                      # dict(x, f, status, nit, violation); control points: bp.control_points(out)
    out = bp.solve(differentiable=True)   # x and f differentiable with respect to the tensors given above
    pos = bp.sample(out, num_points=200)  # [B, d, 200]

Every field of a container is supported: terminal waypoints with velocities, directions, accelerations, zero
velocity or a moving target end, intermediate waypoints (with velocities), all derivative bounds (max / min
velocity, upward / horizontal velocity, acceleration with gravity, jerk, tangential acceleration), one turning bound,
spherical obstacles, safe-flight corridors given by their end points and box paddings.  The parameter-row order is
that of ``pack_problem``: ``assemble_rows`` is checked against it field by field on the CPU
(tests/test_packing.py) and on the GPU (tests/test_batched.py).
"""
import numpy as np

from . import batch as tgb, builder, matrix_evaluation, problem as pk


def _torch():
    import torch
    return torch


def assemble_rows(dimension, start, end, start_velocity=None, end_velocity=None, end_zero_velocity=False,
                  intermediate_locations=None, intermediate_velocities=None, max_velocity=None, max_acceleration=None,
                  turning=None, obstacle_centers=None, obstacle_radii=None, corridor_points=None,
                  intervals_per_corridor=None, objective_function_type="minimal_velocity_and_time_path",
                  num_intervals_free_space=None, start_zero_velocity=False, end_is_target=False, start_direction=None,
                  end_direction=None, start_acceleration=None, end_acceleration=None, min_velocity=None,
                  max_upward_velocity=None, max_horizontal_velocity=None, gravity=None, max_jerk=None,
                  tangential_acceleration=None):
    """Shape descriptor and parameter-row blocks of B problems of one shape, in the order ``problem.pack_problem``
    writes them for one container (TG/trajectory_generator.py:134-250).  Works on tensors of any device (the blocks
    are views / casts of the inputs); the corridor block is a zero placeholder that ``builder.sfc_boxes_batch`` fills.
    Returns (spec, blocks, index of the corridor block or None, intervals per corridor or None).

    What a container decides from its data is a flag here, because the batch shares one shape:
    ``start_zero_velocity`` / ``end_zero_velocity`` (a waypoint whose velocity is zero pins three control points
    and has no derivative rows unless a direction or an acceleration is given), ``end_is_target`` (the end waypoint
    moves with ``end_velocity``); a direction may only be given next to no velocity or a zero velocity
    (DS/waypoint_data.py:47-51)."""
    torch = _torch()
    d = int(dimension)
    if objective_function_type not in pk.OBJECTIVES:
        raise Exception("Error, Invalid objective function type")
    B, dev = start.shape[0], start.device
    col = lambda v: (torch.full((B, 1), float(v), dtype=torch.float64, device=dev) if np.isscalar(v)
                     else v.reshape(B, -1).to(torch.float64))
    niw = 0 if intermediate_locations is None else intermediate_locations.shape[2]
    ncorr = 0 if corridor_points is None else corridor_points.shape[2] - 1
    # ---- sizes (TG/trajectory_generator.py:134-162)
    ipc = None
    if ncorr:
        ipc = [2] * ncorr if intervals_per_corridor is None else [int(v) for v in intervals_per_corridor]
        nint = sum(ipc)
    elif num_intervals_free_space is not None:
        nint = int(num_intervals_free_space)
    else:
        s0, s1 = bool(start_zero_velocity), bool(end_zero_velocity)
        nint = 5 + 2 * int(s0) + 2 * int(s1) + int(s0 and s1)
    N = nint + 3
    spec = np.zeros(pk.SP_COUNT, dtype=np.int32)
    spec[pk.SP_DIM], spec[pk.SP_NCP] = d, N
    spec[pk.SP_OBJECTIVE] = pk.OBJECTIVES.index(objective_function_type)
    # ---- terminal locations
    if end_zero_velocity and end_is_target:
        raise Exception("a target end waypoint moves: it cannot have zero velocity")
    spec[pk.SP_START_KIND] = 1 if start_zero_velocity else 0
    spec[pk.SP_END_KIND] = 1 if end_zero_velocity else (2 if end_is_target else 0)
    par = [col(start), col(end)]
    if end_is_target:
        if end_velocity is None:
            raise Exception("a target end waypoint needs its velocity")
        par.append(col(end_velocity))
    # ---- terminal derivative rows (CF/waypoint_constraints.py:73-120): direction, velocity, acceleration per side
    sides = ((start_zero_velocity, start_direction, start_velocity, start_acceleration,
              pk.SP_START_DIR, pk.SP_START_VEL, pk.SP_START_ACC),
             (end_zero_velocity, end_direction, end_velocity, end_acceleration,
              pk.SP_END_DIR, pk.SP_END_VEL, pk.SP_END_ACC))
    for zero, direction, velocity, acceleration, f_dir, f_vel, f_acc in sides:
        if zero and direction is None and acceleration is None:
            continue                                  # zero-velocity waypoint: no derivative rows
        if direction is not None:
            if velocity is not None and not zero:
                raise Exception("a direction cannot be combined with a non-zero velocity")
            spec[f_dir] = 2 if zero else 1
            par.append(col(direction))
        if velocity is not None and not zero:
            spec[f_vel] = 1
            par.append(col(velocity))
        if acceleration is not None:
            spec[f_acc] = 1
            par.append(col(acceleration))
        if not (spec[f_dir] or spec[f_vel] or spec[f_acc]):
            raise IndexError("terminal waypoint needs a velocity, direction or acceleration")
    if niw:
        spec[pk.SP_NIW] = niw
        par.append(col(intermediate_locations))                     # (d, niw) row-major per problem
        if intermediate_velocities is not None:
            spec[pk.SP_IW_VEL] = 1
            par.append(col(intermediate_velocities))
    # ---- derivative bounds (CF/derivative_constraints.py:17-121); the block exists when one of max velocity, max
    #      acceleration, min velocity, max jerk is set (DS/dynamic_bounds.py: checkIfDerivativesActive)
    for value, what in ((max_upward_velocity, "upward"), (max_horizontal_velocity, "horizontal")):
        if value is not None and max_velocity is None:
            raise Exception("To set max %s velocity you need a general max velocity" % what)
    if any(v is not None for v in (max_velocity, max_acceleration, min_velocity, max_jerk)):
        grav = gravity if max_acceleration is not None else None           # only read next to max_acceleration
        for flag, value in ((pk.SP_DB_MINV, min_velocity), (pk.SP_DB_MAXV, max_velocity),
                            (pk.SP_DB_UP, max_upward_velocity), (pk.SP_DB_HORIZ, max_horizontal_velocity),
                            (pk.SP_DB_MAXA, max_acceleration), (pk.SP_DB_GRAV, grav), (pk.SP_DB_JERK, max_jerk)):
            if value is not None:
                spec[flag] = 1
                par.append(col(value))
    if tangential_acceleration is not None:
        lo, hi = tangential_acceleration
        spec[pk.SP_TANG] = 1
        par += [col(lo), col(hi)]
    if turning is not None:
        spec[pk.SP_TURN] = pk.TURN_KINDS[turning[0]]
        par.append(col(turning[1]))
    i_sfc = None
    if ncorr:
        if ncorr > pk.MAX_CORRIDORS:
            raise Exception("at most %d corridors are supported" % pk.MAX_CORRIDORS)
        spec[pk.SP_NCORR] = ncorr
        spec[pk.SP_IPC0:pk.SP_IPC0 + ncorr] = ipc
        i_sfc = len(par)
        par.append(torch.zeros((B, ncorr * (d * d + 2 * d)), dtype=torch.float64, device=dev))
    if obstacle_centers is not None:
        K = obstacle_centers.shape[1]
        spec[pk.SP_NOBST] = K
        par += [obstacle_centers.transpose(1, 2).reshape(B, -1).to(torch.float64), col(obstacle_radii)]   # c-major
    return spec, par, i_sfc, ipc


class BatchedProblem:
    def __init__(self, dimension, start, end, start_velocity=None, end_velocity=None, end_zero_velocity=False,
                 intermediate_locations=None, intermediate_velocities=None, max_velocity=None, max_acceleration=None,
                 turning=None, obstacle_centers=None, obstacle_radii=None, corridor_points=None, corridor_pads=None,
                 intervals_per_corridor=None, objective_function_type="minimal_velocity_and_time_path",
                 num_intervals_free_space=None, initial_scale_factor=1.0, **more):
        """`more`: the remaining container fields -- start_zero_velocity, end_is_target, start_direction,
        end_direction, start_acceleration, end_acceleration, min_velocity, max_upward_velocity,
        max_horizontal_velocity, gravity, max_jerk, tangential_acceleration=(min, max); see ``assemble_rows``."""
        torch = _torch()
        d = int(dimension)
        if not start.is_cuda:
            raise RuntimeError("BatchedProblem needs CUDA tensors (there is no CPU path)")
        B = start.shape[0]
        spec, par, i_sfc, ipc = assemble_rows(
            d, start, end, start_velocity, end_velocity, end_zero_velocity, intermediate_locations,
            intermediate_velocities, max_velocity, max_acceleration, turning, obstacle_centers, obstacle_radii,
            corridor_points, intervals_per_corridor, objective_function_type, num_intervals_free_space, **more)
        niw, ncorr, N = int(spec[pk.SP_NIW]), int(spec[pk.SP_NCORR]), int(spec[pk.SP_NCP])
        self.spec = spec
        self.layout = pk.Layout(spec)
        self.par = torch.cat(par, 1).contiguous()
        if self.par.shape[1] != self.layout.P:
            raise RuntimeError("parameter rows have %d entries, layout expects %d" % (self.par.shape[1], self.layout.P))
        if ncorr:
            builder.sfc_boxes_batch(spec, corridor_points.to(torch.float64), corridor_pads.to(torch.float64), self.par)
        # ---- initial variables (TG/objectives/objective_variables.py:27-48): along the corridor points, else the waypoints
        wseq = None
        if niw:
            wseq = torch.cat([start.reshape(B, d, 1), intermediate_locations, end.reshape(B, d, 1)], 2).to(torch.float64)
        seq = corridor_points.to(torch.float64) if ncorr else (
            wseq if wseq is not None else torch.stack([start, end], 2).to(torch.float64))
        self.x0 = builder.initial_guess_batch(spec, seq, wseq, initial_scale_factor)
        self.B, self.d, self.N = B, d, N

    def solve(self, jacobian="fd", maxiter=100, ftol=1e-6, differentiable=False):
        """-> dict(x [B,n], f, status, nit, violation) of CUDA tensors (x is a fresh tensor; self.x0 is kept).
        differentiable=True: ``batch.solve_differentiable`` (multipliers and polish included, so the dict also holds
        lam, kkt, polish_status and polish_iters); x and f are then differentiable, and ``backward()`` reaches the
        tensors given to the constructor through the parameter rows -- waypoints, velocities, accelerations,
        directions, bounds given as tensors, obstacle centres and radii.  The corridor block is computed by
        ``builder.sfc_boxes_batch`` outside autograd: no gradient reaches corridor points or pads (``batch.sensitivity``
        still returns the gradient of the corridor entries of the rows)."""
        if differentiable:
            return tgb.solve_differentiable(self.spec, self.par, self.x0, maxiter=maxiter, ftol=ftol, jacobian=jacobian)[2]
        x = self.x0.clone()
        return tgb.solve(self.spec, self.par, x, maxiter=maxiter, ftol=ftol, jacobian=jacobian)

    def control_points(self, out):
        """-> (control_points [B, d, N], scale_factors [B]) views of the solver rows"""
        x = out["x"]
        return x[:, :self.d * self.N].reshape(self.B, self.d, self.N), x[:, self.d * self.N]

    def sample(self, out, num_points=None, dt=None, derivative_order=0):
        return matrix_evaluation.sample_batch((out["x"], self.d, self.N), derivative_order=derivative_order,
                                              num_points=num_points, dt=dt)


class CorridorProblems:
    """Corridor problems whose SHAPE follows from their geometry, as in the reference: ``SFC_Data`` chooses the
    intervals of every corridor from the segment lengths (DS/safe_flight_corridor.py:78-88) and
    ``TrajectoryGenerator`` the number of control points from their sum (TG/trajectory_generator.py:148-162), so a
    batch of raw corridor polylines is a mix of shapes.  Everything happens on the device: intervals per corridor
    (``tg_sfc_intervals_batch``), grouping by shape key (one sort), one ``BatchedProblem`` per shape (boxes, parameter
    rows, initial guess), and ONE solve call for all shapes (``tg_solve_mixed_batch``).

        cp = CorridorProblems(3, corridor_points=pts, corridor_pads=pads, start_velocity=v0, end_zero_velocity=True,
                              max_velocity=5.0, max_acceleration=0.3, objective_function_type="minimal_velocity_path")
        out = cp.solve()      # status / nit / f / violation [B] in input order; out["buckets"]: per shape (indices, problem, x)

    Per-problem tensor arguments (anything with a leading batch axis) are split along with the problems; scalars and
    tuples are shared."""

    def __init__(self, dimension, corridor_points, corridor_pads, min_intervals_per_corridor=1, **fields):
        torch = _torch()
        if not corridor_points.is_cuda:
            raise RuntimeError("CorridorProblems needs CUDA tensors (there is no CPU path)")
        pts = corridor_points.to(torch.float64).contiguous()
        B = pts.shape[0]
        self.B, self.d = B, int(dimension)
        self.ipc, key = builder.sfc_intervals_batch(pts, min_intervals_per_corridor)
        uniq, inverse = torch.unique(key, return_inverse=True)
        order = torch.argsort(inverse, stable=True)
        counts = torch.bincount(inverse, minlength=len(uniq)).cpu().tolist()
        self.buckets = []
        lo = 0
        for cnt in counts:
            idx = order[lo:lo + cnt]
            lo += cnt
            take = lambda v: v[idx] if (torch.is_tensor(v) and v.dim() >= 1 and v.shape[0] == B) else v
            sub = {k: take(v) for k, v in fields.items()}
            ipc = self.ipc[idx[0]].cpu().tolist()
            prob = BatchedProblem(self.d, start=pts[idx][:, :, 0].contiguous(), end=pts[idx][:, :, -1].contiguous(),
                                  corridor_points=pts[idx].contiguous(), corridor_pads=corridor_pads[idx].contiguous(),
                                  intervals_per_corridor=ipc, **sub)
            self.buckets.append((idx, prob))

    def shapes(self):
        """-> list of (intervals per corridor, number of problems), one entry per shape"""
        return [(self.ipc[idx[0]].cpu().tolist(), int(idx.numel())) for idx, _ in self.buckets]

    def solve(self, jacobian="fd", maxiter=100, ftol=1e-6):
        torch = _torch()
        xs = [p.x0.clone() for _, p in self.buckets]
        outs = tgb.solve_mixed([(p.spec, p.par, x) for (_, p), x in zip(self.buckets, xs)], maxiter, ftol, jacobian)
        dev = xs[0].device
        res = dict(status=torch.empty(self.B, dtype=torch.int32, device=dev), nit=torch.empty(self.B, dtype=torch.int32, device=dev),
                   violation=torch.empty(self.B, dtype=torch.int32, device=dev), f=torch.empty(self.B, dtype=torch.float64, device=dev),
                   buckets=[])
        for (idx, prob), out in zip(self.buckets, outs):
            for k in ("status", "nit", "violation", "f"):
                res[k][idx] = out[k]
            res["buckets"].append((idx, prob, out["x"]))
        return res
