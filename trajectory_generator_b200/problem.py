"""Host-side problem packing: ``ConstraintsContainer`` -> (shape descriptor, parameter row, x0, bounds).

Mirrors what ``TrajectoryGenerator.generate_trajectory`` assembles before it calls SLSQP
(reference TG/trajectory_generator.py:65-86, 134-250 and TG/objectives/objective_variables.py:27-105):
number of intervals / control points, the variable vector ``[P row-major | alpha | direction
scalars | intermediate times]``, its bounds and initial guess, and which constraint blocks exist.
The blocks themselves are evaluated on the GPU (csrc/tg_eval.h); here they are reduced to the
int32 descriptor of csrc/tg_spec.h plus one flat float64 parameter row per problem.
"""
import numpy as np

from . import _native

OBJECTIVES = ("minimal_time_path", "minimal_distance_path", "minimal_velocity_path",
              "minimal_acceleration_path", "minimal_distance_and_time_path",
              "minimal_velocity_and_time_path", "minimal_acceleration_and_time_path",
              "minimal_time_path_velocity_penalty")
TURN_KINDS = {"curvature": 1, "angular_rate": 2, "centripetal_acceleration": 3}

# indices into the spec array: keep in step with enum TgSpecField (csrc/tg_spec.h)
MAX_CORRIDORS = 8
(SP_DIM, SP_NCP, SP_OBJECTIVE, SP_START_KIND, SP_END_KIND, SP_START_DIR, SP_START_VEL, SP_START_ACC,
 SP_END_DIR, SP_END_VEL, SP_END_ACC, SP_NIW, SP_IW_VEL, SP_DB_MINV, SP_DB_MAXV, SP_DB_UP, SP_DB_HORIZ,
 SP_DB_MAXA, SP_DB_GRAV, SP_DB_JERK, SP_TANG, SP_TURN, SP_NCORR, SP_IPC0) = range(24)
SP_NOBST = SP_IPC0 + MAX_CORRIDORS
SP_COUNT = SP_NOBST + 1

VARIABLE_LOWER_BOUND = 10e-8     # TG/objectives/objective_variables.py:56 (the literal is 10e-8 = 1e-7)


class Layout:
    """Row / column / parameter offsets derived from a spec (struct TgLayout of csrc/tg_spec.h)."""

    _cache = {}          # spec bytes -> field dict (a batch of containers shares a handful of shapes)

    def __init__(self, spec):
        key = np.ascontiguousarray(spec, dtype=np.int32).tobytes()
        fields = Layout._cache.get(key)
        if fields is None:
            fields = {name: int(value) for name, value in zip(_native.LAYOUT_FIELDS, _native.layout_ints(spec))}
            Layout._cache[key] = fields
        self.__dict__.update(fields)

    # constraint row blocks in SLSQP row order: (name, first-row field, row-count field, kind)
    _ROW_BLOCKS = (("start", "r_start", "n_start", "eq"), ("end", "r_end", "n_end", "eq"),
                   ("start_derivatives", "r_sder", "n_sder", "eq"), ("end_derivatives", "r_eder", "n_eder", "eq"),
                   ("intermediate_locations", "r_iwl", "n_iwl", "eq"), ("intermediate_velocities", "r_iwv", "n_iwv", "eq"),
                   ("derivative_bounds", "r_db", "n_db", "ineq"), ("tangential_lower", "r_tanl", "n_tan", "ineq"),
                   ("tangential_upper", "r_tanu", "n_tan", "ineq"), ("turning", "r_turn", "n_turn", "ineq"),
                   ("corridor_lower", "r_sfcl", "n_sfc", "ineq"), ("corridor_upper", "r_sfcu", "n_sfc", "ineq"),
                   ("obstacles", "r_obs", "n_obs", "ineq"))

    def row_blocks(self):
        """The non-empty constraint row blocks in row order, as (name, start, stop, "eq" | "ineq"): which rows of the
        constraint values and of the multipliers (batch.solve(..., multipliers=True)) belong to which constraint.  They
        tile [0, m); the equality blocks come first and end at meq."""
        out = []
        for name, r, cnt, kind in self._ROW_BLOCKS:
            start, count = getattr(self, r), getattr(self, cnt)
            if count:
                out.append((name, start, start + count, kind))
        return out


class PackedProblem:
    def __init__(self, spec, par, x0, xl, xu):
        self.spec, self.par, self.x0, self.xl, self.xu = spec, par, x0, xl, xu
        self.layout = Layout(spec)

    @property
    def key(self):
        return self.spec.tobytes()


def _flat(a):
    return np.asarray(a, dtype=np.float64).flatten()


def num_intervals_free_space(waypoint_data, requested=None):
    """TG/trajectory_generator.py:134-146."""
    if requested is not None:
        return requested
    s0 = waypoint_data.start_waypoint.checkIfZeroVel()
    s1 = waypoint_data.end_waypoint.checkIfZeroVel()
    return 5 + 2 * int(s0) + 2 * int(s1) + int(s0 and s1)


def initial_control_points(num_cont_pts, point_sequence, dimension):
    """Straight line, or equal arc-length steps along the polyline (TG/objectives/objective_variables.py:63-93)."""
    seq = np.asarray(point_sequence, dtype=np.float64)
    nseg = seq.shape[1] - 1
    if nseg < 2:
        return np.linspace(seq[:, 0], seq[:, 1], num_cont_pts).T
    cps = np.empty((dimension, num_cont_pts))
    cum = np.cumsum(np.linalg.norm(seq[:, 1:] - seq[:, :-1], 2, 0))
    spacing = cum[nseg - 1] / (num_cont_pts - 1)
    seg, walked, anchor, step = 0, 0.0, seq[:, 0], 0.0
    for i in range(num_cont_pts - 1):
        heading = seq[:, seg + 1] - seq[:, seg]
        cps[:, i] = anchor + heading / np.linalg.norm(heading) * step
        anchor = cps[:, i]
        step = spacing
        walked = walked + step
        if cum[seg] < walked:
            step = walked - cum[seg]
            seg += 1
            anchor = seq[:, seg]
    cps[:, -1] = seq[:, -1]
    return cps


def initial_intermediate_times(waypoint_locations, num_cont_pts):
    """TG/objectives/objective_variables.py:95-105."""
    nseg = waypoint_locations.shape[1] - 1
    if nseg <= 2:
        return np.array([0.5])
    cum = np.cumsum(np.linalg.norm(waypoint_locations[:, 1:] - waypoint_locations[:, :-1], 2, 0))
    return (cum / cum[nseg - 1])[:-1] * (num_cont_pts - 3)


PATH_OBJECTIVES = ("minimal_distance_path", "minimal_velocity_path", "minimal_acceleration_path")


def pack_problem(dimension, constraints_container, objective_function_type="minimal_velocity_and_time_path",
                 num_intervals_free_space_arg=None, initial_control_points_arg=None, initial_scale_factor=None,
                 path_mode=None):
    """path_mode None: the problem TrajectoryGenerator.generate_trajectory hands to SLSQP
    (TG/trajectory_generator.py:65-97, 171-250).  path_mode "direct" / "indirect": the problem
    PathGenerator.generate_path builds (TG/path_generator.py:45-82, 145-202): plain location rows at both ends
    whatever the velocities, direction rows only (always the s (P2 - P0) / 2 form), intermediate locations
    without velocities, the curvature bound as the turning row ("direct") or as min velocity 0.5 / max
    acceleration kappa 0.5^2 ("indirect", :177-185), corridors, obstacles; no derivative bounds of the container."""
    d = int(dimension)
    cc = constraints_container
    wd, db, tb = cc.waypoint_constraints, cc.derivative_constraints, cc.turning_constraint
    sfc, obstacles = cc.sfc_constraints, cc.obstacle_constraints
    sw, ew = wd.start_waypoint, wd.end_waypoint
    if path_mode not in (None, "direct", "indirect"):
        raise ValueError("path_mode must be None, 'direct' or 'indirect'")
    if objective_function_type not in (OBJECTIVES if path_mode is None else PATH_OBJECTIVES):
        raise Exception("Error, Invalid objective function type")
    if path_mode is not None:
        return _pack_path_problem(d, cc, objective_function_type, num_intervals_free_space_arg,
                                  initial_control_points_arg, initial_scale_factor, path_mode == "indirect")

    # ---- sizes (TG/trajectory_generator.py:134-162)
    mew0 = num_intervals_free_space(wd, num_intervals_free_space_arg)
    if initial_control_points_arg is not None:
        nint = np.shape(initial_control_points_arg)[1] - 3
    elif sfc is not None:
        nint = sfc.get_num_intervals()
    else:
        nint = mew0
    N = int(nint + 3)

    spec = np.zeros(SP_COUNT, dtype=np.int32)
    spec[SP_DIM], spec[SP_NCP] = d, N
    spec[SP_OBJECTIVE] = OBJECTIVES.index(objective_function_type)
    par = []

    # ---- terminal locations
    spec[SP_START_KIND] = 1 if sw.checkIfZeroVel() else 0
    spec[SP_END_KIND] = 1 if ew.checkIfZeroVel() else (2 if ew.is_target else 0)
    par += [_flat(sw.location), _flat(ew.location)]
    if spec[SP_END_KIND] == 2:
        par.append(_flat(ew.velocity))

    # ---- terminal derivative rows (CF/waypoint_constraints.py:73-120)
    for wp, (f_dir, f_vel, f_acc) in ((sw, (SP_START_DIR, SP_START_VEL, SP_START_ACC)),
                                      (ew, (SP_END_DIR, SP_END_VEL, SP_END_ACC))):
        if not wp.checkIfDerivativesActive():
            continue
        speed = np.linalg.norm(_flat(wp.velocity)) if wp.checkIfVelocityActive() else None
        if wp.checkIfDirectionActive():
            spec[f_dir] = 2 if (speed is not None and speed <= 0) else 1
            par.append(_flat(wp.direction))
        if speed is not None and speed > 0:
            spec[f_vel] = 1
            par.append(_flat(wp.velocity))
        if wp.checkIfAccelerationActive():
            spec[f_acc] = 1
            par.append(_flat(wp.acceleration))
        if not (spec[f_dir] or spec[f_vel] or spec[f_acc]):
            # the reference builds a zero-row NonlinearConstraint here and scipy raises (SURVEY.md fact 10)
            raise IndexError("terminal waypoint needs a velocity, direction or acceleration")

    # ---- intermediate waypoints
    niw = wd.get_num_intermediate_waypoints()
    spec[SP_NIW] = niw
    if niw:
        par.append(_flat(wd.intermediate_locations))
        if wd.intermediate_velocities is not None:
            spec[SP_IW_VEL] = 1
            par.append(_flat(wd.intermediate_velocities))

    # ---- derivative bounds (CF/derivative_constraints.py:17-121)
    if db is not None and db.checkIfDerivativesActive():
        gravity = db.gravity if db.max_acceleration is not None else None      # only read next to max_acceleration
        for flag, value in ((SP_DB_MINV, db.min_velocity), (SP_DB_MAXV, db.max_velocity),
                            (SP_DB_UP, db.max_upward_velocity), (SP_DB_HORIZ, db.max_horizontal_velocity),
                            (SP_DB_MAXA, db.max_acceleration), (SP_DB_GRAV, gravity), (SP_DB_JERK, db.max_jerk)):
            if value is not None:
                spec[flag] = 1
                par.append(np.array([float(value)]))
    if db is not None and db.checkIfTangentialAccelerationActive():
        spec[SP_TANG] = 1
        par.append(np.array([float(db.min_tangential_acceleration), float(db.max_tangential_acceleration)]))

    # ---- turning bound
    if tb is not None and tb.checkIfTurningBoundActive():
        spec[SP_TURN] = TURN_KINDS[tb.bound_type]
        par.append(np.array([float(tb.max_turning_bound)]))

    # ---- safe flight corridors, obstacles
    if sfc is not None:
        par += _corridor_blocks(spec, sfc, nint)
    if obstacles is not None:
        par += _obstacle_blocks(spec, obstacles, d)

    return _finish_packing(d, N, spec, par, wd, sfc, initial_control_points_arg, initial_scale_factor)


def _finish_packing(d, N, spec, par, wd, sfc, initial_control_points_arg, initial_scale_factor):
    """parameter row, initial variables and bounds (TG/objectives/objective_variables.py:27-61)"""
    niw = wd.get_num_intermediate_waypoints()
    par = np.concatenate(par) if par else np.zeros(0)
    packed = PackedProblem(spec, None, None, None, None)
    lay = packed.layout
    if lay.P != par.size:
        raise RuntimeError("parameter row has %d entries, layout expects %d" % (par.size, lay.P))
    n = lay.n
    seq = wd.get_waypoint_locations() if sfc is None else sfc.get_point_sequence()
    if initial_control_points_arg is not None:
        cps = np.asarray(initial_control_points_arg, dtype=np.float64)
    else:
        cps = initial_control_points(N, seq, d)
    x0 = np.empty(n)
    x0[:d * N] = cps.flatten()
    x0[d * N] = 1.0 if initial_scale_factor is None else initial_scale_factor
    x0[d * N + 1:d * N + 1 + lay.nws] = 1.0
    if niw:
        x0[lay.it0:] = initial_intermediate_times(wd.get_waypoint_locations(), N)
    xl = np.full(n, -np.inf)
    xu = np.full(n, np.inf)
    xl[d * N:d * N + 1 + lay.nws] = VARIABLE_LOWER_BOUND
    if niw:
        xl[lay.it0:] = 0.0
        xu[lay.it0:] = N - 3
    packed.par, packed.x0, packed.xl, packed.xu = np.ascontiguousarray(par, dtype=np.float64), x0, xl, xu
    return packed


def _corridor_blocks(spec, sfc, nint):
    """descriptor entries and parameter blocks of the corridors (CF/sfc_constraints.py:7-77)"""
    ipc = sfc.get_intervals_per_corridor()
    ipc = [int(ipc)] if np.ndim(ipc) == 0 else [int(v) for v in ipc]
    if len(ipc) > MAX_CORRIDORS:
        raise Exception("at most %d corridors are supported" % MAX_CORRIDORS)
    if sum(ipc) != nint:
        raise Exception("intervals per corridor do not add up to the number of intervals")
    spec[SP_NCORR] = len(ipc)
    spec[SP_IPC0:SP_IPC0 + len(ipc)] = ipc
    par = []
    for box in sfc.get_sfc_list()[:len(ipc)]:
        lo, hi = box.getRotatedBounds()
        par += [_flat(np.asarray(box.rotation).T), _flat(lo), _flat(hi)]
    return par


def _obstacle_blocks(spec, obstacles, d):
    """CF/obstacle_constraints.py:93-113"""
    spec[SP_NOBST] = len(obstacles)
    centers = np.array([[float(np.asarray(o.center).flatten()[c]) for o in obstacles] for c in range(d)])
    return [centers.flatten(), np.array([float(o.radius) for o in obstacles])]


def _pack_path_problem(d, cc, objective_function_type, num_intervals_free_space_arg, initial_control_points_arg,
                       initial_scale_factor, indirect):
    wd, tb, sfc, obstacles = cc.waypoint_constraints, cc.turning_constraint, cc.sfc_constraints, cc.obstacle_constraints
    sw, ew = wd.start_waypoint, wd.end_waypoint
    # ---- sizes (TG/path_generator.py:104-135: the same rule as the trajectory generator's)
    mew0 = num_intervals_free_space(wd, num_intervals_free_space_arg)
    if initial_control_points_arg is not None:
        nint = np.shape(initial_control_points_arg)[1] - 3
    elif sfc is not None:
        nint = sfc.get_num_intervals()
    else:
        nint = mew0
    N = int(nint + 3)
    spec = np.zeros(SP_COUNT, dtype=np.int32)
    spec[SP_DIM], spec[SP_NCP] = d, N
    spec[SP_OBJECTIVE] = OBJECTIVES.index(objective_function_type)
    # ---- plain location rows at both ends (:148-155), direction rows (:156-165)
    par = [_flat(sw.location), _flat(ew.location)]
    for wp, f_dir in ((sw, SP_START_DIR), (ew, SP_END_DIR)):
        if wp.checkIfDirectionActive():
            if indirect:
                # the reference's indirect direction row divides by the waypoint scalar at the start and cancels it
                # at the end (CF/waypoint_constraints.py:212-217): not one of the row kinds of this library
                raise Exception("isIndirect with a waypoint direction is not supported")
            spec[f_dir] = 1
            par.append(_flat(wp.direction))
    # ---- intermediate locations (:166-170; velocities of intermediate waypoints are not read)
    niw = wd.get_num_intermediate_waypoints()
    spec[SP_NIW] = niw
    if niw:
        par.append(_flat(wd.intermediate_locations))
    # ---- curvature bound (:174-190)
    if tb is not None and tb.checkIfCurvatureBoundActive():
        if indirect:
            min_velocity = 0.5
            spec[SP_DB_MINV] = 1
            par.append(np.array([min_velocity]))
            spec[SP_DB_MAXA] = 1
            par.append(np.array([float(tb.max_turning_bound) * min_velocity ** 2]))
        else:
            spec[SP_TURN] = TURN_KINDS["curvature"]
            par.append(np.array([float(tb.max_turning_bound)]))
    if sfc is not None:
        par += _corridor_blocks(spec, sfc, nint)
    if obstacles is not None:
        par += _obstacle_blocks(spec, obstacles, d)
    return _finish_packing(d, N, spec, par, wd, sfc, initial_control_points_arg, initial_scale_factor)


# --------------------------------------------------------------------------------------------------------------
# Vectorised packing of MANY containers (the batched addition generate_trajectories): containers are grouped by a
# shape key read off their fields without any array arithmetic, and each group is packed with one numpy gather per
# field -- the same descriptor, parameter-row order, initial variables and bounds as pack_problem (checked against
# it container by container in tests/test_packing.py).
# --------------------------------------------------------------------------------------------------------------
def _is_zero(v):
    """velocity given and identically zero (Waypoint.checkIfZeroVel without the norm: early exit on the first entry)"""
    if v is None:
        return False
    for e in np.asarray(v).flat:
        if e != 0:
            return False
    return True


def _shape_key(cc, d):
    """Everything that decides the descriptor, as a hashable tuple (no numpy arithmetic)."""
    wd, db, tb = cc.waypoint_constraints, cc.derivative_constraints, cc.turning_constraint
    sfc, obstacles = cc.sfc_constraints, cc.obstacle_constraints
    key = []
    for wp in (wd.start_waypoint, wd.end_waypoint):
        zero = _is_zero(wp.velocity)
        key.append((wp.direction is not None, wp.velocity is not None, zero, wp.acceleration is not None, bool(wp.is_target)))
    key.append((wd.get_num_intermediate_waypoints(), wd.intermediate_velocities is not None))
    if db is None:
        key.append(None)
    else:
        key.append((db.min_velocity is not None, db.max_velocity is not None, db.max_upward_velocity is not None,
                    db.max_horizontal_velocity is not None, db.max_acceleration is not None, db.gravity is not None,
                    db.max_jerk is not None, db.min_tangential_acceleration is not None and db.max_tangential_acceleration is not None))
    key.append(None if tb is None or tb.max_turning_bound is None else tb.bound_type)
    if sfc is None:
        key.append(None)
    else:
        ipc = getattr(sfc, "_tg_ipc_key", None)          # cached on the object (SFC_Data fixes its intervals at construction)
        if ipc is None:
            raw = sfc.get_intervals_per_corridor()
            ipc = (int(raw),) if np.ndim(raw) == 0 else tuple(int(v) for v in raw)
            try:
                sfc._tg_ipc_key = ipc
            except Exception:
                pass
        key.append(ipc)
    key.append(None if obstacles is None else len(obstacles))
    return tuple(key)


def line_initial_points(start, goal, N):
    """np.linspace(start, goal, N) per problem (TG/objectives/objective_variables.py:63-70) -> [B, d, N]"""
    # numpy.linspace: arange * step + start, except that a zero step in ANY coordinate switches the whole call to
    # (arange / div) * delta + start (numpy/_core/function_base.py: any_step_zero)
    delta = goal - start
    div = N - 1
    step = delta / div
    ar = np.arange(N, dtype=np.float64)[None, None, :]
    cps = ar * step[:, :, None] + start[:, :, None]
    zero = (step == 0).any(1)
    if zero.any():
        cps[zero] = (ar / div) * delta[zero][:, :, None] + start[zero][:, :, None]
    cps[:, :, -1] = goal
    return cps


def polyline_initial_points(seq, N):
    """Equal arc-length steps along a polyline (TG/objectives/objective_variables.py:63-93), batched.
    seq: [B, d, S+1] -> [B, d, N]."""
    B, d, S1 = seq.shape
    S = S1 - 1
    seglen = np.linalg.norm(seq[:, :, 1:] - seq[:, :, :-1], 2, 1)
    cum = np.cumsum(seglen, 1)
    spacing = cum[:, S - 1] / (N - 1)
    rows = np.arange(B)
    seg = np.zeros(B, dtype=np.int64)
    walked = np.zeros(B)
    anchor = seq[:, :, 0].copy()
    step = np.zeros(B)
    cps = np.empty((B, d, N))
    for i in range(N - 1):
        sg = np.minimum(seg, S - 1)
        heading = seq[rows, :, sg + 1] - seq[rows, :, sg]
        heading = heading / np.linalg.norm(heading, 2, 1)[:, None]
        cps[:, :, i] = anchor + heading * step[:, None]
        anchor = cps[:, :, i].copy()
        step = spacing.copy()
        walked = walked + step
        adv = cum[rows, sg] < walked
        step = np.where(adv, walked - cum[rows, sg], step)
        seg = seg + adv
        nxt = seq[rows, :, np.minimum(seg, S)]
        anchor = np.where(adv[:, None], nxt, anchor)
    cps[:, :, -1] = seq[:, :, -1]
    return cps


class PackedGroup:
    """B containers of one shape: spec, par [B, P], x0 [B, n] (clipped to the bounds), xl / xu [n], and the positions
    of the containers in the input list."""

    def __init__(self, indices, spec, par, x0, xl, xu):
        self.indices, self.spec, self.par, self.x0, self.xl, self.xu = indices, spec, par, x0, xl, xu
        self.layout = Layout(spec)


def pack_problems(dimension, containers, objective_function_type="minimal_velocity_and_time_path",
                  num_intervals_free_space_arg=None):
    """-> list of PackedGroup, one per shape, covering every container (default initial guesses)."""
    d = int(dimension)
    if objective_function_type not in OBJECTIVES:
        raise Exception("Error, Invalid objective function type")
    groups = {}
    for i, cc in enumerate(containers):
        groups.setdefault(_shape_key(cc, d), []).append(i)
    out = []
    def col(items):
        """list of B column vectors (d x 1, the form the dataclasses hold) -> [B, d]"""
        items = list(items)
        try:
            a = np.concatenate(items, axis=1)               # fast path: every item is a 2-D float column
            if a.ndim == 2 and a.dtype == np.float64 and a.shape[1] == len(items):
                return np.ascontiguousarray(a.T)
        except Exception:
            pass
        return np.array([np.asarray(v, dtype=np.float64).reshape(-1) for v in items])
    for key, idx in groups.items():
        (s_dir, s_vel, s_zero, s_acc, _), (e_dir, e_vel, e_zero, e_acc, e_target), (niw, iw_vel), dbk, turn, ipc, nobst = key
        group = [containers[i] for i in idx]
        B = len(group)
        wds = [c.waypoint_constraints for c in group]
        sws = [w.start_waypoint for w in wds]
        ews = [w.end_waypoint for w in wds]
        # ---- sizes (TG/trajectory_generator.py:134-162)
        if ipc is not None:
            nint = sum(ipc)
        elif num_intervals_free_space_arg is not None:
            nint = num_intervals_free_space_arg
        else:
            nint = 5 + 2 * int(s_zero) + 2 * int(e_zero) + int(s_zero and e_zero)
        N = int(nint + 3)
        spec = np.zeros(SP_COUNT, dtype=np.int32)
        spec[SP_DIM], spec[SP_NCP] = d, N
        spec[SP_OBJECTIVE] = OBJECTIVES.index(objective_function_type)
        spec[SP_START_KIND] = 1 if s_zero else 0
        spec[SP_END_KIND] = 1 if e_zero else (2 if e_target else 0)
        start = col(w.location for w in sws)
        goal = col(w.location for w in ews)
        par = [start, goal]
        if spec[SP_END_KIND] == 2:
            par.append(col(w.velocity for w in ews))
        # ---- terminal derivative rows (CF/waypoint_constraints.py:73-120), as pack_problem
        for wps, (has_dir, has_vel, zero, has_acc), (f_dir, f_vel, f_acc) in (
                (sws, (s_dir, s_vel, s_zero, s_acc), (SP_START_DIR, SP_START_VEL, SP_START_ACC)),
                (ews, (e_dir, e_vel, e_zero, e_acc), (SP_END_DIR, SP_END_VEL, SP_END_ACC))):
            if not (has_acc or has_dir or not zero):          # Waypoint.checkIfDerivativesActive
                continue
            if has_dir:
                spec[f_dir] = 2 if (has_vel and zero) else 1
                par.append(col(w.direction for w in wps))
            if has_vel and not zero:
                spec[f_vel] = 1
                par.append(col(w.velocity for w in wps))
            if has_acc:
                spec[f_acc] = 1
                par.append(col(w.acceleration for w in wps))
            if not (spec[f_dir] or spec[f_vel] or spec[f_acc]):
                raise IndexError("terminal waypoint needs a velocity, direction or acceleration")
        spec[SP_NIW] = niw
        if niw:
            par.append(col(w.intermediate_locations for w in wds))
            if iw_vel:
                spec[SP_IW_VEL] = 1
                par.append(col(w.intermediate_velocities for w in wds))
        # ---- derivative bounds
        if dbk is not None:
            dbs = [c.derivative_constraints for c in group]
            minv, maxv, up, horiz, maxa, grav, jerk, tang = dbk
            if minv or maxv or maxa or jerk:                  # DerivativeBounds.checkIfDerivativesActive
                for flag, present, name in ((SP_DB_MINV, minv, "min_velocity"), (SP_DB_MAXV, maxv, "max_velocity"),
                                            (SP_DB_UP, up, "max_upward_velocity"), (SP_DB_HORIZ, horiz, "max_horizontal_velocity"),
                                            (SP_DB_MAXA, maxa, "max_acceleration"), (SP_DB_GRAV, grav and maxa, "gravity"),
                                            (SP_DB_JERK, jerk, "max_jerk")):
                    if present:
                        spec[flag] = 1
                        par.append(np.array([[float(getattr(b, name))] for b in dbs]))
            if tang:
                spec[SP_TANG] = 1
                par.append(np.array([[float(b.min_tangential_acceleration), float(b.max_tangential_acceleration)] for b in dbs]))
        if turn is not None:
            spec[SP_TURN] = TURN_KINDS[turn]
            par.append(np.array([[float(c.turning_constraint.max_turning_bound)] for c in group]))
        # ---- corridors (CF/sfc_constraints.py:7-77), obstacles (CF/obstacle_constraints.py:93-113)
        seq = None
        if ipc is not None:
            if len(ipc) > MAX_CORRIDORS:
                raise Exception("at most %d corridors are supported" % MAX_CORRIDORS)
            spec[SP_NCORR] = len(ipc)
            spec[SP_IPC0:SP_IPC0 + len(ipc)] = ipc
            boxes = [c.sfc_constraints.get_sfc_list()[:len(ipc)] for c in group]
            flat = [bx for bl in boxes for bx in bl]
            nc = len(ipc)
            rot = np.transpose(np.array([bx.rotation for bx in flat], dtype=np.float64), (0, 2, 1)).reshape(B, nc, d * d)      # R^T row-major
            tr = col(bx.translation for bx in flat).reshape(B, nc, d)
            half = col(bx.dimensions for bx in flat).reshape(B, nc, d) / 2
            par.append(np.concatenate([rot, tr - half, tr + half], 2).reshape(B, -1))
            seq = np.array([np.asarray(c.sfc_constraints.get_point_sequence(), dtype=np.float64) for c in group])
        if nobst is not None:
            spec[SP_NOBST] = nobst
            obs = [o for c in group for o in c.obstacle_constraints]
            ctr = col(o.center for o in obs).reshape(B, nobst, d)
            par.append(np.transpose(ctr, (0, 2, 1)).reshape(B, -1))
            par.append(np.array([o.radius for o in obs], dtype=np.float64).reshape(B, nobst))
        par = np.ascontiguousarray(np.concatenate(par, 1), dtype=np.float64)
        lay = Layout(spec)
        if lay.P != par.shape[1]:
            raise RuntimeError("parameter rows have %d entries, layout expects %d" % (par.shape[1], lay.P))
        # ---- initial variables and bounds (TG/objectives/objective_variables.py:27-105)
        wseq = None
        if niw:
            wseq = np.concatenate([start[:, :, None], np.array([w.intermediate_locations for w in wds], dtype=np.float64),
                                   goal[:, :, None]], 2)
        if seq is None:
            seq = wseq if wseq is not None else np.stack([start, goal], 2)
        cps = line_initial_points(seq[:, :, 0], seq[:, :, 1], N) if seq.shape[2] == 2 else polyline_initial_points(seq, N)
        n = lay.n
        x0 = np.empty((B, n))
        x0[:, :d * N] = cps.reshape(B, -1)
        x0[:, d * N:d * N + 1 + lay.nws] = 1.0
        if niw:
            if wseq.shape[2] - 1 <= 2:
                x0[:, lay.it0:] = 0.5
            else:
                cum = np.cumsum(np.linalg.norm(wseq[:, :, 1:] - wseq[:, :, :-1], 2, 1), 1)
                x0[:, lay.it0:] = (cum / cum[:, -1:])[:, :-1] * (N - 3)
        xl = np.full(n, -np.inf)
        xu = np.full(n, np.inf)
        xl[d * N:d * N + 1 + lay.nws] = VARIABLE_LOWER_BOUND
        if niw:
            xl[lay.it0:] = 0.0
            xu[lay.it0:] = N - 3
        out.append(PackedGroup(np.asarray(idx), spec, par, np.clip(x0, xl, xu), xl, xu))
    return out
