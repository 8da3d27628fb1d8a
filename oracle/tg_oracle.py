"""TEST INFRASTRUCTURE -- CPU oracle for the optimisation hot path.

numpy restatement of what ``TrajectoryGenerator.generate_trajectory`` hands to
scipy SLSQP (reference TG/trajectory_generator.py:65-97): the variable vector,
bounds, objective and every constraint closure, in the row order SLSQP sees
after scipy's ``new_constraint_to_old`` (scipy/optimize/_constraints.py:506-601),
plus the scipy glue that the reference relies on (2-point finite differences,
``minimize(method='SLSQP')``).  Native steps go through the plain-C oracle
(oracle/native/tg_oracle.c) or, with ``native='ref'``, through the reference's
own C++ compiled unmodified (oracle/_ref).

Only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs may import
this.  The product never does.

Parity status: PINNED.  tests/test_oracle_python.py checks it against fixtures
generated from the real reference (tests/golden/make_golden.py imports the
reference in the build container) and against the gtest golden vectors.

The optimiser arithmetic itself is third-party: scipy (version recorded in
every fixture; 1.18.1 in this image), call site TG/trajectory_generator.py:87-94.
"""
import ctypes
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
_ND = np.ctypeslib.ndpointer(dtype=np.float64, ndim=1, flags="C")

FD_STEP = 1.4901161193847656e-08   # scipy _slsqp_py.py:34 (_epsilon = sqrt(eps))

OBJECTIVES = ("minimal_time_path", "minimal_distance_path", "minimal_velocity_path",
              "minimal_acceleration_path", "minimal_distance_and_time_path",
              "minimal_velocity_and_time_path", "minimal_acceleration_and_time_path",
              "minimal_time_path_velocity_penalty")


# --------------------------------------------------------------------------
# native library (same 24 symbols in oracle/_build, oracle/_ref and the product)
# --------------------------------------------------------------------------
class NativeLib:
    """ctypes binding of the reference's C-ABI (SURVEY.md 8(b) B2)."""

    def __init__(self, path):
        self.path = path
        lib = self.lib = ctypes.CDLL(path)
        self.h = {}
        for D in (2, 3):
            for ctor in ("CrossTermBounds", "DerivativeBounds", "ObstacleConstraints", "ControlPointDerivativeBounds"):
                f = getattr(lib, "%s_%d" % (ctor, D))
                f.restype = ctypes.c_void_p
                self.h[(ctor, D)] = f()
            f = getattr(lib, "get_spline_curvature_bound_%d" % D)
            f.argtypes = [ctypes.c_void_p, _ND, ctypes.c_int]; f.restype = ctypes.c_double
            for nm in ("get_spline_angular_rate_bound", "get_spline_centripetal_acceleration_bound",
                       "find_min_velocity_of_spline"):
                f = getattr(lib, "%s_%d" % (nm, D))
                f.argtypes = [ctypes.c_void_p, _ND, ctypes.c_int, ctypes.c_double]; f.restype = ctypes.c_double
            f = getattr(lib, "getObstaclesConstraintsForSpline_%d" % D)
            f.argtypes = [ctypes.c_void_p, _ND, _ND, ctypes.c_int, _ND, ctypes.c_int]
            f.restype = ctypes.POINTER(ctypes.c_double)
            f = getattr(lib, "getObstacleConstraintsForIntervals_%d" % D)
            f.argtypes = [ctypes.c_void_p, _ND, ctypes.c_int, ctypes.c_double, _ND]
            f.restype = ctypes.POINTER(ctypes.c_double)
            f = getattr(lib, "getObstacleConstraintForSpline_%d" % D)
            f.argtypes = [ctypes.c_void_p, _ND, ctypes.c_int, ctypes.c_double, _ND]; f.restype = ctypes.c_double
            f = getattr(lib, "find_min_velocity_of_bez_vel_cont_pts_%d" % D)
            f.argtypes = [ctypes.c_void_p, _ND, ctypes.c_int]; f.restype = ctypes.c_double

    @staticmethod
    def _flat(a):
        return np.ascontiguousarray(np.asarray(a, dtype=np.float64).flatten())

    def turning_bound(self, kind, cp, alpha):
        D, N = cp.shape
        h = self.h[("CrossTermBounds", D)]
        if kind == "curvature":
            return getattr(self.lib, "get_spline_curvature_bound_%d" % D)(h, self._flat(cp), N)
        nm = "get_spline_angular_rate_bound" if kind == "angular_rate" else "get_spline_centripetal_acceleration_bound"
        return getattr(self.lib, "%s_%d" % (nm, D))(h, self._flat(cp), N, float(alpha))

    def min_velocity(self, cp, alpha):
        D, N = cp.shape
        return getattr(self.lib, "find_min_velocity_of_spline_%d" % D)(self.h[("DerivativeBounds", D)],
                                                                       self._flat(cp), N, float(alpha))

    def obstacle_distances(self, cp, centers, radii):
        D, N = cp.shape
        K = len(radii)
        p = getattr(self.lib, "getObstaclesConstraintsForSpline_%d" % D)(
            self.h[("ObstacleConstraints", D)], self._flat(centers), self._flat(radii), K, self._flat(cp), N)
        return np.array([p[i] for i in range(K)])

    def interval_distances(self, cp, radius, center):
        D, N = cp.shape
        p = getattr(self.lib, "getObstacleConstraintsForIntervals_%d" % D)(
            self.h[("ObstacleConstraints", D)], self._flat(cp), N, float(radius), self._flat(center))
        return np.array([p[i] for i in range(N - 3)])

    def spline_distance(self, cp, radius, center):
        D, N = cp.shape
        return getattr(self.lib, "getObstacleConstraintForSpline_%d" % D)(
            self.h[("ObstacleConstraints", D)], self._flat(cp), N, float(radius), self._flat(center))

    def min_velocity_bezier(self, bez):
        D, n = bez.shape
        return getattr(self.lib, "find_min_velocity_of_bez_vel_cont_pts_%d" % D)(
            self.h[("ControlPointDerivativeBounds", D)], self._flat(bez), n)


_NATIVE = {}


def native(kind="oracle"):
    """kind: 'oracle' (plain-C restatement) or 'ref' (reference C++ compiled unmodified)."""
    if kind not in _NATIVE:
        path = {"oracle": os.path.join(HERE, "_build", "libtg_oracle.so"),
                "ref": os.path.join(HERE, "_ref", "libTrajectoryConstraints.so")}[kind]
        if not os.path.exists(path):
            raise RuntimeError("oracle library %s missing: run `make -C oracle`" % path)
        _NATIVE[kind] = NativeLib(path)
    return _NATIVE[kind]


# --------------------------------------------------------------------------
# constants restated from the reference
# --------------------------------------------------------------------------
# TG/matrix_evaluation.py:245-250
M3 = np.array([[-2, 6, -6, 2], [6, -12, 0, 8], [-6, 6, 6, 2], [2, 0, 0, 0]]) / 12
# TG/matrix_evaluation.py:239-243
M2 = 0.5 * np.array([[1, -2, 1], [-2, 2, 1], [1, 0, 0]])
# TG/control_point_conversions/bspline_to_minvo.py:44-48 (already transposed: Q = C @ P_interval^T)
MINVO3_PY = np.array([[1 / 6, 0.057009542139797595613306102386893, -0.015455156825262485566573649098775, 0],
                      [2 / 3, 0.66657381574108923111064205020873, 0.2918717989443756838876956809183, 1 / 6],
                      [1 / 6, 0.2918717989443756838876956809183, 0.66657381574108923111064205020873, 2 / 3],
                      [0, -0.015455156825262485566573649098775, 0.057009542139797595613306102386893, 1 / 6]]).T


def _fact(k):
    return float(np.prod(np.arange(1, k + 1))) if k > 0 else 1.0


def eval_point(cp, t, tj, alpha):
    """TG/matrix_evaluation.py:183-188, 224-232."""
    order = cp.shape[1] - 1
    M = M3 if order == 3 else M2
    T = np.array([((t - tj) / alpha) ** (order - i) for i in range(order + 1)])
    return cp @ M @ T


def eval_derivative(cp, t, tj, alpha, r):
    """TG/matrix_evaluation.py:190-195, 216-222."""
    order = cp.shape[1] - 1
    M = M3 if order == 3 else M2
    T = np.zeros(order + 1)
    for i in range(order - r + 1):
        T[i] = ((t - tj) ** (order - r - i)) / (alpha ** (order - i)) * _fact(order - i) / _fact(order - i - r)
    return cp @ M @ T


def bezier_velocity_matrix(num_vel_pts):
    """TG/control_point_conversions/bspline_to_bezier.py:23-45 for order 2."""
    seg = num_vel_pts - 2
    C = np.zeros((2 * seg + 1, num_vel_pts))
    blk = np.array([[1, 1, 0], [0, 2, 0], [0, 1, 1]]) / 2
    for i in range(seg):
        C[2 * i:2 * i + 3, i:i + 3] = blk
    return C


# --------------------------------------------------------------------------
# problem assembly
# --------------------------------------------------------------------------
class Block:
    """One reference constraint (TG/trajectory_generator.py:171-250) with scipy-style bounds."""

    def __init__(self, name, fun, lb, ub, linear_A=None):
        self.name, self.fun, self.linear_A = name, fun, linear_A
        self.lb, self.ub = lb, ub


class OracleProblem:
    def __init__(self, dimension, container, objective="minimal_velocity_and_time_path",
                 num_intervals_free_space=None, initial_control_points=None, initial_scale_factor=None,
                 native_kind="oracle"):
        self.nat = native(native_kind)
        self.d = d = dimension
        wd = container.waypoint_constraints
        db = container.derivative_constraints
        tb = container.turning_constraint
        obstacles = container.obstacle_constraints
        sfc = container.sfc_constraints
        self.wd, self.db, self.tb, self.obstacles, self.sfc = wd, db, tb, obstacles, sfc
        sw, ew = wd.start_waypoint, wd.end_waypoint
        # TG/trajectory_generator.py:134-162
        if num_intervals_free_space is not None:
            mew0 = num_intervals_free_space
        else:
            mew0 = 5 + 2 * sw.checkIfZeroVel() + 2 * ew.checkIfZeroVel() + (sw.checkIfZeroVel() and ew.checkIfZeroVel())
        if initial_control_points is not None:
            nint = np.shape(initial_control_points)[1] - 3
        elif sfc is not None:
            nint = sfc.get_num_intervals()
        else:
            nint = mew0
        self.N = N = int(nint + 3)
        self.nint = self.N - 3
        self.niw = wd.get_num_intermediate_waypoints()
        self.nws = wd.get_num_waypoint_scalars()
        self.n = d * N + 1 + self.nws + self.niw
        self.objective = objective
        if objective not in OBJECTIVES:
            raise Exception("Error, Invalid objective function type")
        self.point_sequence = wd.get_waypoint_locations() if sfc is None else sfc.get_point_sequence()
        self.xl, self.xu = self._bounds()
        self.x0 = self._initial_variables(initial_control_points, initial_scale_factor)
        self.blocks = self._blocks()
        self._split_rows()

    # ---- TG/objectives/objective_variables.py:50-61 ----
    def _bounds(self):
        lo = np.full(self.n, -np.inf); hi = np.full(self.n, np.inf)
        s = self.d * self.N
        lo[s:s + self.nws + 1] = 10e-8
        if self.niw > 0:
            hi[-self.niw:] = self.N - 3
            lo[-self.niw:] = 0
        return lo, hi

    # ---- TG/objectives/objective_variables.py:27-48, 63-105 ----
    def _initial_variables(self, icp, isf):
        d, N = self.d, self.N
        seq = self.point_sequence
        nseg = seq.shape[1] - 1
        if icp is not None:
            cps = np.asarray(icp, dtype=float)
        elif nseg < 2:
            cps = np.linspace(seq[:, 0], seq[:, 1], N).T
        else:
            cps = np.empty((d, N))
            dist = np.cumsum(np.linalg.norm(seq[:, 1:] - seq[:, :-1], 2, 0))
            step_len = dist[nseg - 1] / (N - 1)
            seg = 0; travelled = 0.0; prev = seq[:, 0]; step = 0.0
            for i in range(N - 1):
                a, b = seq[:, seg], seq[:, seg + 1]
                u = (b - a) / np.linalg.norm(b - a)
                cps[:, i] = prev + u * step
                prev = cps[:, i]
                step = step_len
                travelled = travelled + step
                if dist[seg] < travelled:
                    step = travelled - dist[seg]
                    seg += 1
                    prev = seq[:, seg]
            cps[:, -1] = seq[:, -1]
        alpha = 1 if isf is None else isf
        x = np.concatenate((cps.flatten(), [alpha]))
        if self.wd.start_waypoint.direction is not None:
            x = np.concatenate((x, [1]))
        if self.wd.end_waypoint.direction is not None:
            x = np.concatenate((x, [1]))
        if self.niw > 0:
            wseq = self.wd.get_waypoint_locations()
            nws = wseq.shape[1] - 1
            times = np.array([0.5])
            if nws > 2:
                dist = np.cumsum(np.linalg.norm(wseq[:, 1:] - wseq[:, :-1], 2, 0))
                times = (dist / dist[nws - 1])[:-1] * (N - 3)
            x = np.concatenate((x, times))
        return np.asarray(x, dtype=float)

    # ---- helpers ----
    def cps(self, x):
        return np.reshape(x[:self.d * self.N], (self.d, self.N))

    def alpha(self, x):
        return x[self.d * self.N]

    # ---- TG/objectives/objective_functions.py:6-62 ----
    def fun(self, x):
        P = self.cps(x); a = self.alpha(x)
        D1 = P[:, :-1] - P[:, 1:]
        D2 = P[:, 2:] - 2 * P[:, 1:-1] + P[:, :-2]
        D3 = P[:, 3:] - 3 * P[:, 2:-1] + 3 * P[:, 1:-2] - P[:, :-3]
        ss = lambda D: np.sum(np.sum(D ** 2, 0))
        o = self.objective
        if o == "minimal_time_path": return a ** 2
        if o == "minimal_distance_path": return ss(D1)
        if o == "minimal_velocity_path": return ss(D2)
        if o == "minimal_acceleration_path": return ss(D3)
        if o == "minimal_distance_and_time_path": return ss(D1) * a
        if o == "minimal_velocity_and_time_path": return ss(D2) * a
        if o == "minimal_acceleration_and_time_path": return ss(D3) * a
        return 100 * a ** 2 - ss(D1)

    # ---- constraint blocks in the reference's list order ----
    def _blocks(self):
        d, N, n = self.d, self.N, self.n
        wd = self.wd
        sw, ew = wd.start_waypoint, wd.end_waypoint
        blocks = []

        def loc_rows(side):   # CF/waypoint_constraints.py:10-44
            A = np.zeros((d, n))
            w = M3 @ (np.array([0, 0, 0, 1.0]) if side == "start" else np.ones(4))
            for i in range(d):
                if side == "start": A[i, i * N:i * N + 4] = w
                else: A[i, (i + 1) * N - 4:(i + 1) * N] = w
            return A

        def zero_vel_rows(side):   # CF/waypoint_constraints.py:46-71
            A = np.zeros((3 * d, n))
            for i in range(d):
                c0 = i * N if side == "start" else (i + 1) * N - 3
                A[3 * i:3 * i + 3, c0:c0 + 3] = np.eye(3)
            return A

        for wp, side in ((sw, "start"), (ew, "end")):
            if wp.checkIfZeroVel():
                A = zero_vel_rows(side); b = np.repeat(wp.location.flatten(), 3)
            elif side == "end" and wp.is_target:   # CF/waypoint_constraints.py:122-147
                A = loc_rows("end"); A[:, N * d] = -(N - 3) * wp.velocity.flatten(); b = wp.location.flatten()
            else:
                A = loc_rows(side); b = wp.location.flatten()
            blocks.append(Block(side + "_location", (lambda x, A=A: A @ x), b, b, linear_A=A))
        for wp, side in ((sw, "start"), (ew, "end")):
            if wp.checkIfDerivativesActive():
                f = self._terminal_derivative_fun(wp, side)
                blocks.append(Block(side + "_derivatives", f, 0, 0))
        if wd.intermediate_locations is not None:
            blocks.append(Block("iw_locations", self._iw_location_fun(), 0, 0))
            if wd.intermediate_velocities is not None:
                blocks.append(Block("iw_velocities", self._iw_velocity_fun(), 0, 0))
        db = self.db
        if db is not None and db.checkIfDerivativesActive():
            f, length = self._derivative_fun()
            blocks.append(Block("derivative", f, np.full(length, -np.inf), np.zeros(length)))
        if db is not None and db.checkIfTangentialAccelerationActive():
            blocks.append(Block("tangential", self._tangential_fun(), db.min_tangential_acceleration,
                                db.max_tangential_acceleration))
        tb = self.tb
        if tb is not None and tb.checkIfTurningBoundActive():
            blocks.append(Block("turning", self._turning_fun(), -np.inf, 0))
        if self.sfc is not None:
            A, lo, hi = self._sfc_rows()
            blocks.append(Block("sfc", (lambda x, A=A: A @ x), lo, hi, linear_A=A))
        if self.obstacles is not None:
            K = len(self.obstacles)
            blocks.append(Block("obstacles", self._obstacle_fun(), np.zeros(K), np.full(K, np.inf)))
        return blocks

    # ---- CF/waypoint_constraints.py:73-120, 205-245 ----
    def _terminal_derivative_fun(self, wp, side):
        d, N = self.d, self.N
        dir_on, vel_on, acc_on = wp.checkIfDirectionActive(), wp.checkIfVelocityActive(), wp.checkIfAccelerationActive()
        vmag = np.linalg.norm(wp.velocity.flatten()) if vel_on else None
        s0 = d * N + 1
        length = d * (int(dir_on) + int(vel_on and vmag > 0) + int(acc_on))

        def f(x):
            P = self.cps(x); a = self.alpha(x)
            first, mid, last = (P[:, 0], P[:, 1], P[:, 2]) if side == "start" else (P[:, -3], P[:, -2], P[:, -1])
            out = np.zeros(length); k = 0
            if dir_on:
                scalars = x[s0:s0 + self.nws]
                s = scalars[0] if side == "start" else scalars[-1]
                if vmag is not None and vmag <= 0:
                    far = (P[:, 3] - P[:, 0]) if side == "start" else (P[:, -1] - P[:, -4])
                    direction = s * far / 2
                else:
                    direction = s * (last - first) / 2
                out[k:k + d] = direction - wp.direction.flatten(); k += d
            if vel_on and vmag > 0:
                out[k:k + d] = (last - first) / (2 * a) - wp.velocity.flatten(); k += d
            if acc_on:
                out[k:k + d] = (first - 2 * mid + last) / (a * a) - wp.acceleration.flatten()
            return out
        return f

    # ---- CF/waypoint_constraints.py:248-270 ----
    def _iw_location_fun(self):
        locs = self.wd.intermediate_locations
        d, niw = self.d, self.niw

        def f(x):
            P = self.cps(x); times = x[-niw:]
            out = np.zeros((d, niw))
            for i in range(niw):
                k = int(times[i])
                out[:, i] = eval_point(P[:, k:k + 4], times[i], k, 1) - locs[:, i]
            return out.flatten()
        return f

    # ---- CF/waypoint_constraints.py:272-295 ----
    def _iw_velocity_fun(self):
        vels = self.wd.intermediate_velocities
        d, niw = self.d, self.niw

        def f(x):
            P = self.cps(x); a = self.alpha(x); times = x[-niw:]
            out = np.zeros((d, niw))
            for i in range(niw):
                k = int(times[i])
                t_ = (times[i] - k) * a
                out[:, i] = eval_derivative(P[:, k:k + 4], t_, 0, a, 1) - vels[:, i]
            return out.flatten()
        return f

    # ---- CF/derivative_constraints.py:17-121 ----
    def _derivative_fun(self):
        db, d, N = self.db, self.d, self.N
        Mv = bezier_velocity_matrix(N - 1)
        length = (int(db.min_velocity is not None) + int(db.max_velocity is not None)
                  + int(db.max_velocity is not None and db.max_upward_velocity is not None)
                  + int(db.max_velocity is not None and db.max_horizontal_velocity is not None)
                  + int(db.max_acceleration is not None) + int(db.max_jerk is not None))

        def f(x):
            P = self.cps(x); a = self.alpha(x)
            V = (P[:, 1:] - P[:, :-1]) / a
            out = np.zeros(length); k = 0
            if db.min_velocity is not None or db.max_velocity is not None:
                bez = (Mv @ V.T).T
                if db.min_velocity is not None:
                    out[k] = db.min_velocity - self.nat.min_velocity(P, a); k += 1
                if db.max_velocity is not None:
                    out[k] = np.max(np.linalg.norm(bez, 2, 0)) - db.max_velocity; k += 1
                    if db.max_upward_velocity is not None and d == 3:
                        out[k] = -np.min(bez[2, :]) - db.max_upward_velocity; k += 1
                    if db.max_horizontal_velocity is not None and d == 3:
                        out[k] = np.max(np.linalg.norm(bez[0:2, :], 2, 0)) - db.max_horizontal_velocity; k += 1
            if db.max_acceleration is not None or db.max_jerk is not None:
                A = (V[:, 1:] - V[:, :-1]) / a
                if db.max_acceleration is not None:
                    Ag = A
                    if db.gravity is not None and d == 3:
                        Ag = A - np.array([[0], [0], [db.gravity]])
                    out[k] = np.max(np.linalg.norm(Ag, 2, 0)) - db.max_acceleration; k += 1
                if db.max_jerk is not None:
                    J = (A[:, 1:] - A[:, :-1]) / a
                    out[k] = np.max(np.linalg.norm(J, 2, 0)) - db.max_jerk; k += 1
            return out
        return f, length

    # ---- CF/derivative_constraints.py:124-241 ----
    def _tangential_fun(self):
        nint = self.nint

        def quad_roots(a_, b_, c_):
            with np.errstate(all="ignore"):
                disc = b_ * b_ - 4 * a_ * c_
                if disc == 0:
                    return np.array([np.float64(-b_) / np.float64(2 * a_), np.inf])
                if disc < 0:
                    return np.array([np.inf, np.inf])
                return np.array([(-b_ + np.sqrt(disc)) / np.float64(2 * a_), (-b_ - np.sqrt(disc)) / np.float64(2 * a_)])

        def dot_term(cp, a, t):
            return np.dot(eval_derivative(cp, t, 0, a, 2), eval_derivative(cp, t, 0, a, 1))

        def f(x):
            P = self.cps(x); a = self.alpha(x)
            out = np.zeros((2, nint))
            for i in range(nint):
                cp = P[:, i:i + 4]
                D3 = cp[:, 0] - 3 * cp[:, 1] + 3 * cp[:, 2] - cp[:, 3]
                D2 = cp[:, 0] - 2 * cp[:, 1] + cp[:, 2]
                D1 = cp[:, 0] / 2 - cp[:, 2] / 2
                c2 = np.dot(D3, D3 / 2) + np.dot(D3, D3)
                c1 = -np.dot(3 * D2, D3)
                c0 = np.dot(D2, D2) + np.dot(D1, D3)
                roots = quad_roots(c2, c1, c0)
                hi = lo = dot_term(cp, a, 0)
                with np.errstate(all="ignore"):
                    for t in (roots[0] * a, roots[1] * a, a):
                        if t < 0 or t > a:
                            continue
                        v = dot_term(cp, a, t)
                        if v > hi: hi = v
                        if v < lo: lo = v
                    vmin = self.nat.min_velocity(cp, a)
                    out[0, i] = np.float64(hi) / np.float64(vmin)
                    out[1, i] = np.float64(lo) / np.float64(vmin)
            return out.flatten()
        return f

    # ---- CF/turning_constraints.py:49-121 ----
    def _turning_fun(self):
        tb, wd = self.tb, self.wd

        def f(x):
            P = self.cps(x)
            if wd.start_waypoint.checkIfZeroVel(): P = P[:, 1:]
            if wd.end_waypoint.checkIfZeroVel(): P = P[:, :-1]
            P = np.ascontiguousarray(P)
            b = self.nat.turning_bound(tb.bound_type, P, self.alpha(x))
            with np.errstate(all="ignore"):
                if tb.bound_type == "curvature":
                    return np.array([b - tb.max_turning_bound]) * 100
                return np.array([b - tb.max_turning_bound])
        return f

    # ---- CF/sfc_constraints.py:7-77 ----
    def _sfc_rows(self):
        d, N, n = self.d, self.N, self.n
        nint = N - 3
        npts = 4 * nint
        comp = np.zeros((npts, N))
        for j in range(nint):
            comp[4 * j:4 * j + 4, j:j + 4] = MINVO3_PY
        big = np.zeros((d * npts, n))
        for c in range(d):
            big[c * npts:(c + 1) * npts, c * N:(c + 1) * N] = comp
        ipc = self.sfc.get_intervals_per_corridor()
        sfcs = self.sfc.get_sfc_list()
        if np.ndim(ipc) == 0:
            ipc = [int(ipc)]
        Mrot = np.zeros((d * npts, d * npts))
        lo = np.zeros((d, npts)); hi = np.zeros((d, npts))
        idx = 0
        for ci in range(len(ipc)):
            RT = np.asarray(sfcs[ci].rotation).T
            lb, ub = sfcs[ci].getRotatedBounds()
            for _ in range(int(ipc[ci])):
                for k in range(4):
                    for r in range(d):
                        for c in range(d):
                            Mrot[r * npts + idx, c * npts + idx] = RT[r, c]
                    lo[:, idx] = np.asarray(lb).flatten(); hi[:, idx] = np.asarray(ub).flatten()
                    idx += 1
        return Mrot @ big, lo.flatten(), hi.flatten()

    # ---- CF/obstacle_constraints.py:93-113 ----
    def _obstacle_fun(self):
        obs, d = self.obstacles, self.d
        radii = np.array([float(o.radius) for o in obs])
        centers = np.array([[float(np.asarray(o.center)[c, 0]) for o in obs] for c in range(d)])

        def f(x):
            return self.nat.obstacle_distances(np.ascontiguousarray(self.cps(x)), centers, radii)
        return f

    # ---- scipy _constraints.py:541-580 + _slsqp_py.py:328-372: row triage ----
    def _split_rows(self):
        self.eq_parts, self.ineq_parts = [], []
        for b in self.blocks:
            y0 = np.atleast_1d(b.fun(self.x0))
            lb = np.broadcast_to(np.asarray(b.lb, dtype=float), y0.shape).copy()
            ub = np.broadcast_to(np.asarray(b.ub, dtype=float), y0.shape).copy()
            i_eq = lb == ub
            below = np.logical_xor(lb != -np.inf, i_eq)
            above = np.logical_xor(ub != np.inf, i_eq)
            if np.any(i_eq):
                self.eq_parts.append((b, i_eq, lb))
            if np.sum(below) + np.sum(above):
                self.ineq_parts.append((b, below, above, lb, ub))
        self.meq = sum(int(np.sum(p[1])) for p in self.eq_parts)
        self.mineq = sum(int(np.sum(p[1]) + np.sum(p[2])) for p in self.ineq_parts)
        self.m = self.meq + self.mineq
        # which SLSQP rows come from linear blocks
        lin = []
        for b, i_eq, _ in self.eq_parts:
            lin += [b.linear_A is not None] * int(np.sum(i_eq))
        for b, below, above, _, _ in self.ineq_parts:
            lin += [b.linear_A is not None] * int(np.sum(below) + np.sum(above))
        self.row_is_linear = np.array(lin, dtype=bool)

    def cons(self, x):
        """Constraint vector as SLSQP sees it: meq rows (== 0) then mineq rows (>= 0)."""
        out = []
        cache = {}

        def val(b):
            if id(b) not in cache:
                cache[id(b)] = np.atleast_1d(np.array(b.fun(x), dtype=float)).flatten()
            return cache[id(b)]
        for b, i_eq, lb in self.eq_parts:
            out.append(val(b)[i_eq] - lb[i_eq])
        for b, below, above, lb, ub in self.ineq_parts:
            y = val(b)
            with np.errstate(all="ignore"):
                out.append(y[below] - lb[below])
                out.append(-(y[above] - ub[above]))
        return np.concatenate(out) if out else np.zeros(0)

    def linear_jacobian(self):
        """Constant rows (SLSQP order, SLSQP sign) of the linear blocks; NaN rows elsewhere."""
        J = np.full((self.m, self.n), np.nan)
        r = 0
        for b, i_eq, _ in self.eq_parts:
            k = int(np.sum(i_eq))
            if b.linear_A is not None:
                J[r:r + k] = b.linear_A[i_eq]
            r += k
        for b, below, above, _, _ in self.ineq_parts:
            kb, ka = int(np.sum(below)), int(np.sum(above))
            if b.linear_A is not None:
                J[r:r + kb] = b.linear_A[below]
                J[r + kb:r + kb + ka] = -b.linear_A[above]
            r += kb + ka
        return J

    # ---- scipy _numdiff.py approx_derivative('2-point', abs_step=eps, bounds) ----
    def _fd_steps(self, x):
        h = np.full(self.n, FD_STEP)
        xp = x + h
        violated = (xp < self.xl) | (xp > self.xu)
        fitting = np.abs(h) <= np.maximum(x - self.xl, self.xu - x)
        h[violated & fitting] *= -1
        return h

    def jac_fd(self, x, fun=None):
        """Forward-difference Jacobian exactly as scipy forms it for the reference."""
        fun = self.cons if fun is None else fun
        x = np.clip(np.asarray(x, dtype=float), self.xl, self.xu)
        f0 = np.atleast_1d(fun(x))
        h = self._fd_steps(x)
        J = np.zeros((len(f0), self.n))
        for i in range(self.n):
            x1 = x.copy(); x1[i] += h[i]
            dx = x1[i] - x[i]
            with np.errstate(all="ignore"):
                J[:, i] = (np.atleast_1d(fun(x1)) - f0) / dx
        return J

    def grad_fd(self, x):
        return self.jac_fd(x, fun=lambda z: np.atleast_1d(self.fun(z)))[0]

    def jac_central(self, x, fun=None, h=1e-4, order=4, cols=None):
        """Jacobian oracle: central differences of the oracle closures, 4th order (5-point stencil) or 6th order
        (7-point stencil).  Only meaningful where the active branches are stable over the whole stencil.
        cols: the columns to difference (default all); the result has one column per entry of cols."""
        fun = self.cons if fun is None else fun
        x = np.asarray(x, dtype=float)
        cols = np.arange(self.n) if cols is None else np.asarray(cols, dtype=int)
        m = len(np.atleast_1d(fun(x)))
        J = np.zeros((m, len(cols)))
        weights = {4: ((1, 8.0 / 12), (2, -1.0 / 12)), 6: ((1, 45.0 / 60), (2, -9.0 / 60), (3, 1.0 / 60))}[order]
        for col, i in enumerate(cols):
            hh = h * max(1.0, abs(x[i]))
            e = np.zeros(self.n); e[i] = hh
            with np.errstate(all="ignore"):
                acc = 0.0
                for k, w in weights:
                    acc = acc + w * (np.atleast_1d(fun(x + k * e)) - np.atleast_1d(fun(x - k * e)))
                J[:, col] = acc / hh
        return J

    def jacobian_error(self, J, x, fun=None, cols=None):
        """Element-wise relative error of J against the Jacobian oracle, and the mask of entries the oracle can
        vouch for.  Two independent 6th-order estimates (h = 1e-3 and 2.5e-4) must agree with each other to 1e-10
        for an entry to be trusted: where they do not, a stencil straddles a kink of the reference's piecewise
        smooth closures (max/min over intervals, hull points, root in/out of the interval; SURVEY.md 8(c)) and no
        finite-difference oracle exists for that entry.  cols: check only these columns of J (default all); the
        results then have one column per entry of cols."""
        if cols is not None:
            J = np.asarray(J)[..., cols]
        est = [self.jac_central(x, fun=fun, h=h, order=6, cols=cols) for h in (1e-3, 2.5e-4)]
        with np.errstate(all="ignore"):
            scale = np.maximum(1.0, np.abs(est[1]))
            trusted = np.abs(est[0] - est[1]) <= 1e-10 * scale
            err = np.abs(J - est[1]) / scale
        err = np.where(np.isfinite(err), err, np.where(trusted, np.inf, 0.0))
        return err, trusted

    # ---- TG/trajectory_generator.py:252-275, DS/constraint_function_data.py:12,45-48 ----
    def is_violation(self, x, success=False):
        """The reference's third return value: False after a successful solve; otherwise the loop over the
        constraint list overwrites the flag every time, so only the LAST constraint decides -- any output of it
        outside [lb - 10e-6, ub + 10e-6]."""
        if success or not self.blocks:
            return False
        b = self.blocks[-1]
        y = np.atleast_1d(np.array(b.fun(np.asarray(x, dtype=float)), dtype=float)).flatten()
        with np.errstate(all="ignore"):
            return bool(np.any((y > np.asarray(b.ub, dtype=float) + 10e-6) | (y < np.asarray(b.lb, dtype=float) - 10e-6)))

    # ---- TG/trajectory_generator.py:85-97 through scipy ----
    def scipy_constraints(self):
        """The old-style dicts scipy builds from the reference's constraint tuple."""
        cons = []
        for b, i_eq, lb in self.eq_parts:
            cons.append({"type": "eq", "fun": (lambda x, b=b, i=i_eq, l=lb: np.atleast_1d(np.array(b.fun(x), dtype=float)).flatten()[i] - l[i])})
            if b.linear_A is not None:
                cons[-1]["jac"] = (lambda x, A=b.linear_A[i_eq]: A)
        for b, below, above, lb, ub in self.ineq_parts:
            def f(x, b=b, below=below, above=above, lb=lb, ub=ub):
                y = np.atleast_1d(np.array(b.fun(x), dtype=float)).flatten()
                return np.concatenate((y[below] - lb[below], -(y[above] - ub[above])))
            cons.append({"type": "ineq", "fun": f})
            if b.linear_A is not None:
                cons[-1]["jac"] = (lambda x, A=np.vstack((b.linear_A[below], -b.linear_A[above])): A)
        return cons

    def solve(self, maxiter=100, ftol=1e-6):
        """scipy SLSQP exactly as the reference calls it (FD Jacobians, default options)."""
        from scipy.optimize import minimize, Bounds
        import warnings
        with warnings.catch_warnings(), np.errstate(all="ignore"):
            warnings.simplefilter("ignore")
            res = minimize(self.fun, x0=self.x0, method="SLSQP", bounds=Bounds(lb=self.xl, ub=self.xu),
                           constraints=self.scipy_constraints(), options={"disp": False, "maxiter": maxiter, "ftol": ftol})
        return res
