/*
 * C-ABI of the B200-native trajectory_generator hot path.
 *
 * One shared library, libTrajectoryConstraints.so, exports
 *   (A) the reference's own 24 extern "C" symbols, so that it can be dropped at the
 *       path the reference's ctypes wrappers load
 *       (CF/TrajectoryConstraintsCCode/build/src/libTrajectoryConstraints.so;
 *        CF = trajectory_generation/constraint_functions), and
 *   (B) batched entry points for the whole inner loop of
 *       TrajectoryGenerator.generate_trajectory (TG/trajectory_generator.py:65-97):
 *       objective + constraints + analytic Jacobians (what scipy SLSQP calls each
 *       iteration) and the SLSQP iteration itself, one warp per problem.
 *
 * Everything runs on the current CUDA device; there is no CPU fallback: every entry
 * point returns a non-zero status (and tg_last_error() a message) if no device /
 * kernel image is available.
 *
 * Conventions (same as the reference, CC/src/CBindHelperFunctions.cpp:11-31):
 * control points are row-major D x N float64.  Batched arrays are row-major with the
 * problem index slowest.  `spec` is a host array of tg_spec_count() ints (see
 * trajectory_generator_b200/csrc/tg_spec.h) describing the shape shared by all
 * problems of a batch; `par` holds one parameter row of layout.P doubles per problem.
 */
#ifndef TRAJECTORY_GENERATOR_B200_H
#define TRAJECTORY_GENERATOR_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------ (B) batched API */

/* number of ints in a spec / in the layout struct */
int tg_spec_count(void);
/* fills out[] with struct TgLayout (all ints, field order of tg_spec.h); returns its length */
int tg_layout(const int *spec, int *out, int cap);
/* index (1..) of the kernel instantiation with a compile-time descriptor that serves `spec` (the BASELINE.json
 * shapes, csrc/tg_shape.h), 0 when the shape runs the generic kernels.  Results are bit-identical either way. */
int tg_fixed_shape_index(const int *spec);
/* message of the last failing call on this thread ("" if none) */
const char *tg_last_error(void);
/* 0 when a CUDA device with an sm_100a image is usable, else an error code */
int tg_device_check(void);

/*
 * M1: one evaluation of everything scipy SLSQP asks of the reference's closures:
 *   f[B], g[B*n] = objective and gradient           (TG/objectives/objective_functions.py:6-62)
 *   c[B*m]       = constraint rows in SLSQP order   (scipy/optimize/_constraints.py:506-601)
 *   jnl[B*m_nl*n]= Jacobian rows of the nonlinear rows (dense, row-major)
 * replaces per problem: 1 + (n+1) calls of the objective and of every constraint closure
 * (TG/trajectory_generator.py:171-250; scipy 2-point finite differences).
 * Device pointers; any output pointer may be NULL.  `stream` is a cudaStream_t (NULL = default).
 */
int tg_eval_batch(const int *spec, int B, const double *par, const double *x,
                  double *f, double *g, double *c, double *jnl, void *stream);

/* constant Jacobian of the linear rows, all m rows x n (nonlinear rows left untouched): alin[B*m*n] */
int tg_linear_rows_batch(const int *spec, int B, const double *par, double *alin, void *stream);

/* flags for tg_solve_batch */
#define TG_SOLVE_FD_JACOBIAN 1   /* emulate scipy's forward differences (h = 1.4901161193847656e-08) */
#define TG_SOLVE_FUSED 2         /* one persistent kernel (a warp runs a whole solve) instead of lock-step stage kernels */

/* bytes of device scratch tg_solve_batch needs for this shape and batch size */
size_t tg_solve_workspace_bytes(const int *spec, int B);
/* launch plan of the lock-step solve for this shape and batch size on the current device: out[0..6] = {lanes per problem
 * of the line-search stage, lanes per problem of the QP stage, state staged in shared memory by the QP stage, QP
 * scratch in global memory, line-search / derivative scratch in global memory, workspace slots, KiB of the slots}.
 * Scratch goes to global memory (one workspace slot per resident lane group) only for shapes whose scratch does not
 * fit in shared memory, or under the A/B switches TG_QP_FAR=1 / TG_LS_FAR=1.  Returns the number of values, or the
 * negated error code (see tg_last_error). */
int tg_solve_plan_info(const int *spec, int B, int *out, int cap);

/*
 * M2: the per-problem scipy.optimize.minimize(method='SLSQP', options={'disp': False})
 * call of TG/trajectory_generator.py:87-94, batched.  x[B*n]: in = initial variables
 * (TG/objectives/objective_variables.py:27-48), out = optimised variables.
 * status[B] = SLSQP exit mode (0 ok, 4/6 subproblem failures, 8, 9), nit[B] = major iterations,
 * violation[B] = the reference's is_violation flag (TG/trajectory_generator.py:252-261),
 * f[B] = final objective.  Device pointers.
 */
int tg_solve_batch(const int *spec, int B, const double *par, double *x, double *f,
                   int *status, int *nit, int *violation, int maxiter, double ftol, int flags,
                   void *workspace, size_t workspace_bytes, void *stream);
/*
 * tg_solve_batch plus, unless NULL, per problem:
 *   lam[B*m]  the KKT multipliers of the last QP in constraint row order (scipy's OptimizeResult.multipliers: the
 *             equality rows, then the inequality rows; no bound multipliers).  The terminal location rows, which the
 *             QP eliminates, get theirs from the QP's stationarity on the eliminated coordinates (csrc/tg_sqp.h,
 *             tg_sqp_kkt).  For status != 0 they are the last successful QP's values.
 *   kkt[B*4]  first-order optimality certificate at the returned x, absolute, NaN = +inf, with the derivatives the
 *             solve used (analytic or finite-difference) and gradL = g - sum_j lam_j grad c_j:
 *             [0] stationarity max_i |gradL_i| (only its infeasible sign at a variable on its bound),
 *             [1] infeasibility max |c_j| (equality rows), max(0, -c_j) (inequality rows),
 *             [2] dual infeasibility max(0, -lam_j), [3] complementarity max |lam_j c_j| (inequality rows).
 * x, f, status, nit and violation are those of tg_solve_batch.
 */
int tg_solve_batch_kkt(const int *spec, int B, const double *par, double *x, double *f,
                       int *status, int *nit, int *violation, int maxiter, double ftol, int flags,
                       void *workspace, size_t workspace_bytes, void *stream, double *lam, double *kkt);

/* host-buffer variants: copy in, launch, copy out (the reference-facing call measured as `e2e`) */
int tg_eval_host(const int *spec, int B, const double *par, const double *x,
                 double *f, double *g, double *c, double *jnl);
int tg_solve_host(const int *spec, int B, const double *par, double *x, double *f,
                  int *status, int *nit, int *violation, int maxiter, double ftol, int flags);

/*
 * Problems of DIFFERENT shapes in one call (SURVEY.md 8(f) f3).  The reference derives the number of control
 * points and the corridor split of every problem from its geometry (TG/trajectory_generator.py:148-162,
 * DS/safe_flight_corridor.py:78-88), so a set of ConstraintsContainers is a mix of shapes; the caller groups
 * them into `nbuckets` buckets by shape descriptor.  specs = nbuckets x tg_spec_count() ints; counts[k] problems
 * in bucket k; par[k], x[k], f[k], status[k], nit[k], violation[k] = that bucket's HOST arrays, laid out as for
 * tg_solve_host (f / status / nit / violation, or single entries of them, may be NULL).  Buckets are solved
 * concurrently, each on its own stream; results are those of tg_solve_host on every bucket.
 */
int tg_solve_mixed_host(int nbuckets, const int *specs, const int *counts, const double *const *par,
                        double *const *x, double *const *f, int *const *status, int *const *nit,
                        int *const *violation, int maxiter, double ftol, int flags);
/* the same with DEVICE pointers (par[k], x[k], f[k], ... are device buffers; the array of pointers itself is a host
 * array): the buckets run on internal streams that fork from and join `stream`; nothing is copied */
int tg_solve_mixed_batch(int nbuckets, const int *specs, const int *counts, const double *const *par, double *const *x,
                         double *const *f, int *const *status, int *const *nit, int *const *violation, int maxiter,
                         double ftol, int flags, void *stream);
/* the same with tg_solve_batch_kkt's outputs: lam[k] (counts[k] * m of bucket k) and kkt[k] (counts[k] * 4) are device
 * buffers; lam, kkt or any entry of them may be NULL */
int tg_solve_mixed_batch_kkt(int nbuckets, const int *specs, const int *counts, const double *const *par,
                             double *const *x, double *const *f, int *const *status, int *const *nit,
                             int *const *violation, int maxiter, double ftol, int flags, void *stream,
                             double *const *lam, double *const *kkt);

/*
 * Multi-start solves: K seeded starts per problem, solved as ordinary problems, the best one kept.  The problems are
 * non-convex and SLSQP converges to the basin its start lies in; several starts find better basins.  A multi-start
 * solve of B problems is three calls on one stream:
 *   tg_multistart_expand  par[B*P], x0[B*n] -> par_out[B*K*P], x_out[B*K*n]: row b*K + k is start k of problem b.
 *       par_out rows are copies of par[b].  Start 0 is x0[b] bit for bit (K = 1 is an ordinary solve).  Start k > 0
 *       offsets the interior control points (3 .. N-4 of each coordinate) by spread * |P_{N-1} - P_0| times a smooth
 *       profile drawn from a splitmix64 hash of (seed, k, coordinate, knot), and multiplies the scale factor by
 *       1, 1/2, 2, 3/4, 3/2, 5/8, 5/4, 3 (k mod 8); waypoint scalars and intermediate times are copied
 *       (csrc/tg_multistart.cu).  The starts depend on (seed, k) and on the problem itself, never on b.
 *   tg_solve_batch / tg_solve_mixed_batch on the B*K rows, unchanged.
 *   tg_multistart_select  per problem, the constraint rows at each start's final point xs[B*K*n] are folded into the
 *       true maximum violation (max |c| over the equality rows, max(0, -c) over the inequality rows, NaN = +inf;
 *       written to max_violation[B*K] unless it is NULL).  The winner: a start with status 0 and maximum violation
 *       <= tol beats every other start, the lowest f among them (NaN = +inf); with no such start, the lowest maximum
 *       violation, then the lowest f; remaining ties go to the lowest k.  Its x / f / status / nit / violation are
 *       gathered into x_best[B*n], f_best[B], status_best[B], nit_best[B], violation_best[B] (violation stays the
 *       reference's is_violation flag) and best_start[b] = k.  par[B*P] are the B problems' rows.
 * Device pointers; K >= 1.  Returns 0, or an error code with tg_last_error() (K < 1, NULL required pointer, no device).
 */
int tg_multistart_expand(const int *spec, int B, int K, const double *par, const double *x0, unsigned long long seed,
                         double spread, double *par_out, double *x_out, void *stream);
int tg_multistart_select(const int *spec, int B, int K, const double *par, const double *xs, const double *f,
                         const int *status, const int *nit, const int *violation, double tol, double *x_best,
                         double *f_best, int *status_best, int *nit_best, int *violation_best, int *best_start,
                         double *max_violation, void *stream);

/*
 * Output sampling of a batch of cubic trajectories (SURVEY.md 8(f) f1), device pointers:
 *   mode 0: matrix_bspline_evaluation_for_dataset / matrix_bspline_derivative_evaluation_for_dataset
 *           (TG/matrix_evaluation.py:5-33, 104-135): num_points samples over the N-3 intervals of every trajectory;
 *   mode 1: matrix_bspline_evaluation_for_discrete_steps / ..._derivative_evaluation_for_discrete_steps
 *           (TG/matrix_evaluation.py:66-102, 137-173): samples every dt from offset[b] (NULL = 0); counts[b] receives
 *           the number of samples of trajectory b, times[b*capacity + k] (optional) the reference's time_data
 *           before start_time is added.
 * Trajectory b: control points row-major d x N at cps + b*cps_stride, scale factor at scale[b*scale_stride]
 * (so the solver's variable rows x[B][n] can be passed as they are: cps = x, cps_stride = n, scale = x + d*N).
 * out[(b*d + c)*capacity + k]: coordinate c of sample k, the layout of the reference's spline_data[d, num_points].
 * derivative_order 0..3.
 */
int tg_sample_batch(int d, int N, int B, const double *cps, long cps_stride, const double *scale, long scale_stride,
                    int derivative_order, int mode, int num_points, const double *offset, double dt,
                    double *out, long capacity, double *times, int *counts, void *stream);

/* the same for B-splines of order 2 .. 5 (the reference's get_M_matrix, TG/matrix_evaluation.py:197-262;
 * tg_sample_batch is order 3); derivative_order <= order */
int tg_sample_batch_order(int order, int d, int N, int B, const double *cps, long cps_stride, const double *scale,
                          long scale_stride, int derivative_order, int mode, int num_points, const double *offset,
                          double dt, double *out, long capacity, double *times, int *counts, void *stream);

/*
 * One point (or r-th derivative) of one spline interval per item -- evaluate_point_on_interval /
 * evaluate_point_derivative_on_interval (TG/matrix_evaluation.py:183-195), the primitive of the reference's waypoint
 * closures: out[b][c] = cps[b][c][0..order] . M . T(t[b], tj[b], scale[b]).  cps[B][d][order+1], device pointers.
 */
int tg_interval_points_batch(int order, int d, int B, const double *cps, const double *t, const double *tj,
                             const double *scale, int derivative_order, double *out, void *stream);

/*
 * Shape from geometry (SURVEY.md 8(f) f2 -> f3): intervals per corridor as SFC_Data chooses them
 * (DS/safe_flight_corridor.py:78-88) from the corridor end points[B][d][ncorr+1]; ipc[B][ncorr], key[B] (optional) =
 * the ipc values packed 8 bits each, equal for problems of one shape.  Device pointers.
 */
int tg_sfc_intervals_batch(int d, int ncorr, int B, const double *points, int min_per_corridor, int *ipc,
                           long long *key, void *stream);

/*
 * Spline order converter (SURVEY.md 8(f) f4; SmoothingSpline.generate_new_control_points,
 * TG/spline_order_converter.py:22-34): for every old spline, control points x[b][d][N] of a B-spline of `order` that
 * minimise the squared distance to the old spline over `resolution` samples with position, velocity and acceleration
 * matched at both ends, solved with the batched SLSQP iteration (finite-difference gradient as scipy forms it).
 *   par[b] = [Y (d x resolution: samples of the old spline) | b (d x 6: old position at t0, t1, velocity, acceleration)]
 *   x: in = initial control points (tg_smooth_initial_batch: the arc-length walk of create_initial_control_points,
 *      :83-112; scratch = B * oldN doubles), out = solution.  d * N <= 160.  Device pointers.
 */
size_t tg_smooth_workspace_bytes(int d, int N, int order, int resolution, int B);
int tg_smooth_batch(int d, int N, int order, int resolution, double scale, int B, const double *par, double *x,
                    double *f, int *status, int *nit, int maxiter, double ftol, void *workspace, size_t workspace_bytes,
                    void *stream);
int tg_smooth_initial_batch(int d, int oldN, int N, int B, const double *old_cps, double *x0, double *scratch, void *stream);

/*
 * Problem construction on the device (SURVEY.md 8(f) f2), device pointers:
 *   tg_initial_guess_batch: x0[B][n] = [control points | scale0 | waypoint scalars (1) | intermediate times] as
 *     create_initial_objective_variables builds them (TG/objectives/objective_variables.py:27-48, 63-105) from the
 *     point sequence seq[B][d][npts] (2 points: straight line; more: equal arc-length steps along the polyline) and,
 *     with intermediate waypoints, the waypoint locations wseq[B][d][nwp] (nwp = niw + 2).
 *   tg_sfc_boxes_batch: fits one box per corridor to consecutive points[B][d][ncorr+1]
 *     (get2D/3DRotationAndTranslationFromPoints, DS/safe_flight_corridor.py:109-146; dimensions = pad[B][ncorr][d]
 *     + (segment length, 0, 0); SFC.getRotatedBounds, :13-16) and writes [R^T | lower | upper] into the corridor
 *     slots of the parameter rows par[B][P]; lengths[B][ncorr] (optional) receives the segment lengths.
 */
int tg_initial_guess_batch(const int *spec, int B, const double *seq, int npts, const double *wseq, int nwp,
                           double scale0, double *x0, void *stream);
int tg_sfc_boxes_batch(const int *spec, int B, const double *points, const double *pad, double *par,
                       double *lengths, void *stream);

/* number of kernel launches issued by this library since load (all entry points) */
unsigned long long tg_launch_count(void);

/* ---- measurement helpers (bench.py's roofline; not part of the reference's interface)
 * tg_set_stage_timing(1): the following lock-step solves record CUDA events around every stage launch.
 * tg_last_solve_stats: out[0..5] = {ms in line-search launches, ms in QP launches, model fp64 operation count of
 *   the QP stage summed over the batch, line-search launches, QP launches, rounds} of the calling thread's last
 *   solve with timing on; returns the number of values.
 * tg_measure_fp64_peak: DFMA throughput of the current device in TFLOP/s (8 independent chains per thread). */
void tg_set_stage_timing(int on);
int tg_last_solve_stats(double *out, int cap);
int tg_measure_fp64_peak(double *tflops);

/* ------------------------------------------------------------------ (A) legacy symbols
 * Signatures of CC/include/CrossTermBounds.hpp:45-72, CC/include/ObstacleConstraints.hpp:25-49,
 * CC/include/DerivativeBounds.hpp:63-70 and CC/include/ControlPointDerivativeBounds.hpp:26-33
 * (CC = CF/TrajectoryConstraintsCCode).  Host pointers; each call is one single-problem
 * kernel launch.  Returned double* buffers stay valid until the next call on the same
 * handle (the reference leaks them; scipy copies immediately). */
#define TG_DECLARE_LEGACY(D)                                                                                     \
    void *CrossTermBounds_##D(void);                                                                             \
    double get_spline_curvature_bound_##D(void *obj, double cont_pts[], int num_control_points);                 \
    double get_spline_angular_rate_bound_##D(void *obj, double cont_pts[], int num_control_points,               \
                                             double scale_factor);                                               \
    double get_spline_centripetal_acceleration_bound_##D(void *obj, double cont_pts[], int num_control_points,   \
                                                         double scale_factor);                                   \
    void *DerivativeBounds_##D(void);                                                                            \
    double find_min_velocity_of_spline_##D(void *obj, double cont_pts[], int num_control_points,                 \
                                           double scale_factor);                                                 \
    void *ObstacleConstraints_##D(void);                                                                         \
    double *getObstaclesConstraintsForSpline_##D(void *obj, double obstacle_centers[], double obstacle_radii[],  \
                                                 int num_obstacles, double cont_pts[], int num_cont_points);     \
    double *getObstacleConstraintsForIntervals_##D(void *obj, double cont_pts[], int num_cont_points,            \
                                                   double obstacle_radius, double obstacle_center[]);            \
    double getObstacleConstraintForSpline_##D(void *obj, double cont_pts[], int num_cont_points,                 \
                                              double obstacle_radius, double obstacle_center[]);                 \
    void *ControlPointDerivativeBounds_##D(void);                                                                \
    double find_min_velocity_of_bez_vel_cont_pts_##D(void *obj, double cont_pts[], int num_control_points);

TG_DECLARE_LEGACY(2)
TG_DECLARE_LEGACY(3)

#ifdef __cplusplus
}
#endif
#endif /* TRAJECTORY_GENERATOR_B200_H */
