// Objective, constraint and ANALYTIC Jacobian evaluation of one trajectory
// problem -- the functions scipy SLSQP calls on every iteration of
// TrajectoryGenerator.generate_trajectory (reference TG/trajectory_generator.py:87-94).
//
// One warp evaluates one problem.  Work items (intervals, obstacle x interval
// pairs, Bezier points, rows) are strided over the 32 lanes; max/min terms are
// folded with warp shuffles.  The same source compiles for the host with one
// "lane" (TG_NL == 1); that build exists only for the CPU test harness under
// tests/hostsim and is never loaded by the product.
//
// x, par must be readable by every lane (shared memory on the device).
// Constraint rows are in SLSQP order (tg_spec.h).  Every inequality row is in
// the ">= 0" form scipy hands to SLSQP.
//
// The reference has no analytic derivatives (SURVEY.md fact 1); the Jacobians
// here differentiate the reference's closures at the active branch (active
// interval / extremum time / hull point), which is what its finite differences
// approximate away from kinks.
#ifndef TG_EVAL_H
#define TG_EVAL_H

#include <float.h>
#include <math.h>
#include "tg_spec.h"

#define TG_PI 3.14159265358979323846

// TG_HD (tg_spec.h) force-inlines small helpers; TG_FN is for the large block evaluators.  A translation
// unit may define TG_INLINE_ALL (kernels in which every warp runs the same code: inlining pays) -- the
// solver stages keep them out of line (instruction-cache footprint).
#if defined(__CUDACC__)
#if defined(TG_INLINE_ALL)
#define TG_FN static __host__ __device__ inline
#else
#define TG_FN static __host__ __device__ __noinline__
#endif
#else
#define TG_FN static inline
#endif
// the cubic solver (two call sites per interval evaluation) stays out of line in the solver's kernels: one copy
// keeps the code of a finite-difference sweep within reach of the instruction cache
#if defined(__CUDACC__) && !defined(TG_INLINE_LEAVES)
#define TG_LEAF static __host__ __device__ __noinline__
#else
#define TG_LEAF TG_FN
#endif

// translation units that call the whole-problem evaluators from several places (the solver's line-search stage:
// evaluation, finite-difference sweep) define TG_SHARED_EVALUATORS: one out-of-line copy instead of one per call site
#if defined(__CUDACC__) && defined(TG_SHARED_EVALUATORS)
#define TG_EVAL_FN static __host__ __device__ __noinline__
#else
#define TG_EVAL_FN TG_FN
#endif

// A problem is evaluated by a GROUP of TG_GS consecutive lanes of a warp (TG_GS = 8, 16 or 32, fixed per
// translation unit): with 5..14 intervals per spline a full warp leaves most lanes idle in the per-interval
// terms, so several problems share a warp.  Syncs and shuffles only involve the lanes of the group.
#ifndef TG_GS
#define TG_GS 32
#endif
// TG_GS == 64 (QP stage of shapes with more than 32 variables): a group is two consecutive warps; its barrier is
// the named barrier 1 + group index and its folds go through a few shared-memory slots.
#define TG_MAX_CTA_GROUPS64 4
#if defined(__CUDA_ARCH__)
#define TG_LANE() ((int)(threadIdx.x & (TG_GS - 1)))
#define TG_NL TG_GS
#if TG_GS == 64
#define TG_GMASK() 0xffffffffu
#define TG_SYNC() asm volatile("bar.sync %0, 64;" ::"r"((int)(threadIdx.x >> 6) + 1) : "memory")
#else
#define TG_GMASK() (TG_GS == 32 ? 0xffffffffu : (((1u << (TG_GS & 31)) - 1u) << ((threadIdx.x & 31u) & ~(unsigned)(TG_GS - 1))))
#define TG_SYNC() __syncwarp(TG_GMASK())
#endif
#else
#define TG_LANE() 0
#define TG_NL 1
#define TG_SYNC() ((void)0)
#endif
// Serial recurrences with a group sync per step (back substitutions, the forward substitution of the factor update):
// a 64-lane group runs them on its first warp alone -- a warp sync per step instead of a named barrier between two
// warps -- and meets at one TG_SYNC() afterwards.  Same arithmetic, same order.
#if defined(__CUDA_ARCH__) && TG_GS == 64
#define TG_SERIAL_LANES 32
#define TG_SERIAL_ACTIVE() (TG_LANE() < 32)
#define TG_SERIAL_SYNC() __syncwarp()
#else
#define TG_SERIAL_LANES TG_NL
#define TG_SERIAL_ACTIVE() true
#define TG_SERIAL_SYNC() TG_SYNC()
#endif

// ---------------------------------------------------------------------------
// group folds (identity on the host build)
// ---------------------------------------------------------------------------
// (The folds as functions of their own -- one copy each instead of ~100 inlined copies of 10 .. 20 shuffles -- were
// measured on the 32-lane QP kernels, whose warps wait on instruction fetch: QP stage +6 ... 8 %, the calls cost more
// than the fetches they save.)
TG_HD double tg_wsum(double v)
{
#if defined(__CUDA_ARCH__)
#pragma unroll
    for (int o = (TG_GS > 32 ? 32 : TG_GS) / 2; o > 0; o >>= 1) v += __shfl_xor_sync(TG_GMASK(), v, o);
#if TG_GS == 64
    __shared__ double slot[TG_MAX_CTA_GROUPS64][2];
    const int g = threadIdx.x >> 6;
    if ((threadIdx.x & 31) == 0) slot[g][(threadIdx.x >> 5) & 1] = v;
    TG_SYNC();
    v = slot[g][0] + slot[g][1];
    TG_SYNC();
#endif
#endif
    return v;
}

// two sums at once: same folds, but a 64-lane group exchanges both partial sums through shared memory behind ONE pair of
// named barriers instead of two
TG_HD void tg_wsum2(double &a, double &b)
{
#if defined(__CUDA_ARCH__)
#pragma unroll
    for (int o = (TG_GS > 32 ? 32 : TG_GS) / 2; o > 0; o >>= 1) {
        a += __shfl_xor_sync(TG_GMASK(), a, o);
        b += __shfl_xor_sync(TG_GMASK(), b, o);
    }
#if TG_GS == 64
    __shared__ double slot[TG_MAX_CTA_GROUPS64][2][2];
    const int g = threadIdx.x >> 6;
    if ((threadIdx.x & 31) == 0) { slot[g][(threadIdx.x >> 5) & 1][0] = a; slot[g][(threadIdx.x >> 5) & 1][1] = b; }
    TG_SYNC();
    a = slot[g][0][0] + slot[g][1][0];
    b = slot[g][0][1] + slot[g][1][1];
    TG_SYNC();
#endif
#endif
}

// larger value wins; ties -> smaller index (the reference scans upward with a strict '>')
TG_HD void tg_wargmax(double &v, int &i)
{
#if defined(__CUDA_ARCH__)
#pragma unroll
    for (int o = (TG_GS > 32 ? 32 : TG_GS) / 2; o > 0; o >>= 1) {
        double ov = __shfl_xor_sync(TG_GMASK(), v, o);
        int oi = __shfl_xor_sync(TG_GMASK(), i, o);
        if (ov > v || (ov == v && oi < i)) { v = ov; i = oi; }
    }
#if TG_GS == 64
    __shared__ double sv[TG_MAX_CTA_GROUPS64][2];
    __shared__ int si[TG_MAX_CTA_GROUPS64][2];
    const int g = threadIdx.x >> 6;
    if ((threadIdx.x & 31) == 0) { sv[g][(threadIdx.x >> 5) & 1] = v; si[g][(threadIdx.x >> 5) & 1] = i; }
    TG_SYNC();
    v = sv[g][0]; i = si[g][0];
    if (sv[g][1] > v || (sv[g][1] == v && si[g][1] < i)) { v = sv[g][1]; i = si[g][1]; }
    TG_SYNC();
#endif
#endif
}

TG_HD void tg_wargmin(double &v, int &i)
{
#if defined(__CUDA_ARCH__)
#pragma unroll
    for (int o = (TG_GS > 32 ? 32 : TG_GS) / 2; o > 0; o >>= 1) {
        double ov = __shfl_xor_sync(TG_GMASK(), v, o);
        int oi = __shfl_xor_sync(TG_GMASK(), i, o);
        if (ov < v || (ov == v && oi < i)) { v = ov; i = oi; }
    }
#if TG_GS == 64
    __shared__ double sv[TG_MAX_CTA_GROUPS64][2];
    __shared__ int si[TG_MAX_CTA_GROUPS64][2];
    const int g = threadIdx.x >> 6;
    if ((threadIdx.x & 31) == 0) { sv[g][(threadIdx.x >> 5) & 1] = v; si[g][(threadIdx.x >> 5) & 1] = i; }
    TG_SYNC();
    v = sv[g][0]; i = si[g][0];
    if (sv[g][1] < v || (sv[g][1] == v && si[g][1] < i)) { v = sv[g][1]; i = si[g][1]; }
    TG_SYNC();
#endif
#endif
}

TG_HD double tg_bcast(double v, int src)
{
#if defined(__CUDA_ARCH__)
#if TG_GS == 64
    __shared__ double slot[TG_MAX_CTA_GROUPS64];
    const int g = threadIdx.x >> 6;
    if (TG_LANE() == src) slot[g] = v;
    TG_SYNC();
    v = slot[g];
    TG_SYNC();
    return v;
#else
    return __shfl_sync(TG_GMASK(), v, src, TG_GS);
#endif
#else
    (void)src;
    return v;
#endif
}

TG_HD int tg_any(int pred)
{
#if defined(__CUDA_ARCH__)
#if TG_GS == 64
    __shared__ int slot[TG_MAX_CTA_GROUPS64][2];
    const int g = threadIdx.x >> 6;
    const int a = __any_sync(0xffffffffu, pred) != 0;
    if ((threadIdx.x & 31) == 0) slot[g][(threadIdx.x >> 5) & 1] = a;
    TG_SYNC();
    const int r = slot[g][0] | slot[g][1];
    TG_SYNC();
    return r;
#else
    return __any_sync(TG_GMASK(), pred) != 0;
#endif
#else
    return pred != 0;
#endif
}

// ---------------------------------------------------------------------------
// Jacobian sink.  Element (row r, column i) lives at p[row(r) * rs + i * cs].
// compact == 1: only nonlinear rows are stored, re-indexed densely (the M1
// output layout); compact == 0: every row r is stored; compact == 2: every row
// except the corridor rows, the rows behind them moved up (the SQP's A matrix:
// a corridor normal has 4 d structural non-zeros that are regenerated from the
// corridor's rotation and the MINVO matrix where they are needed, tg_sqp.h).
// ---------------------------------------------------------------------------
struct TgJac {
    double *p;
    int rs, cs, compact;
};

TG_HD int tg_nlrow(const TgLayout &L, int r)
{
    const int lin0 = L.n_start + L.n_end;
    if (r < L.r_sder) return -1;
    if (r < L.r_sfcl) return r - lin0;
    if (r < L.r_obs) return -1;
    return r - lin0 - 2 * L.n_sfc;
}

TG_HD double *tg_jrow(const TgJac &J, const TgLayout &L, int r)
{
    // rows in front of the corridor block (compact == 2 stores them unmoved); rows behind it go through tg_jrow_hi
    return J.p + (J.compact == 1 ? tg_nlrow(L, r) : r) * J.rs;
}

// row r >= L.r_obs (behind the corridor block)
TG_HD double *tg_jrow_hi(const TgJac &J, const TgLayout &L, int r)
{
    return J.p + (J.compact == 1 ? tg_nlrow(L, r) : J.compact == 2 ? r - 2 * L.n_sfc : r) * J.rs;
}

// ---------------------------------------------------------------------------
// cubic solver, CC/src/CubicEquationSolver.cpp:8-117 (absent roots = DBL_MAX)
// ---------------------------------------------------------------------------
TG_LEAF void tg_solve_cubic_eq(double a, double b, double c, double d, double r[3])
{
    r[0] = r[1] = r[2] = DBL_MAX;
    if (a == 0) {
        if (b == 0) {
            if (c != 0) r[0] = -d / c;
            return;
        }
        double disc = c * c - 4 * b * d;
        if (disc == 0) r[0] = -c / (2 * b);
        else if (disc > 0) {
            double sq = sqrt(disc);
            r[0] = (-c + sq) / (2 * b);
            r[1] = (-c - sq) / (2 * b);
        }
        return;
    }
    const double disc = 18 * a * b * c * d - 4 * (b * b * b) * d + (b * b) * (c * c) - 4 * a * (c * c * c) -
                        27 * (a * a) * (d * d);
    if (disc > 0) {
        const double ba = b / a, ca = c / a, da = d / a;
        const double Q = (3 * ca - ba * ba) / 9;
        const double R = (9 * ba * ca - 27 * da - 2 * (ba * ba * ba)) / 54;
        const double mq = -Q, sq = sqrt(mq);
        const double theta = acos(R / (mq * sq));
        r[0] = 2 * sq * cos(theta / 3) - ba / 3;
        r[1] = 2 * sq * cos((theta + 2 * TG_PI) / 3) - ba / 3;
        r[2] = 2 * sq * cos((theta + 4 * TG_PI) / 3) - ba / 3;
    } else if (disc < 0) {
        const double P = b * b - 3 * a * c;
        const double Q = 9 * a * b * c - 2 * (b * b * b) - 27 * (a * a) * d;
        const double sq = sqrt((Q * Q) / 4 - P * P * P);
        const double N = cbrt(Q / 2 + sq) + cbrt(Q / 2 - sq);
        r[0] = -b / (3 * a) + N / (3 * a);
    } else {
        const double P = b * b - 3 * a * c;
        if (P == 0) r[0] = -b / (3 * a);
        else {
            r[0] = (9 * a * d - b * c) / (2 * P);
            r[1] = (4 * a * b * c - 9 * a * a * d - b * b * b) / (a * P);
        }
    }
}

// ---------------------------------------------------------------------------
// one cubic B-spline interval: p(tau) = k3 tau^3 + k2 tau^2 + k1 tau + k0 with
// (k3 k2 k1 k0) = P M, M from CC/src/DerivativeEvaluator.cpp:56-65 ==
// TG/matrix_evaluation.py:245-250.  C3/C2/C1 are the columns of M.
// ---------------------------------------------------------------------------
template <int D>
struct TgInterval {
    double k3[D], k2[D], k1[D];
};

#define TG_C3(l) ((l) == 0 ? -1.0 / 6.0 : (l) == 1 ? 0.5 : (l) == 2 ? -0.5 : 1.0 / 6.0)
#define TG_C2(l) ((l) == 0 ? 0.5 : (l) == 1 ? -1.0 : (l) == 2 ? 0.5 : 0.0)
#define TG_C1(l) ((l) == 0 ? -0.5 : (l) == 2 ? 0.5 : 0.0)

// control points of interval j out of the row-major d x N block of x
// (CC/src/CBindHelperFunctions.cpp:11-31); `first` trims the window.
// (pi, pv): entry pi of x is read as pv -- a finite-difference perturbation applied on load.
#define TG_XP(idx) ((idx) == pi ? pv : x[idx])
template <int D>
TG_HD void tg_load_interval(const double *x, int N, int j, TgInterval<D> &I, int pi = -1, double pv = 0)
{
#pragma unroll
    for (int c = 0; c < D; c++) {
        const double p0 = TG_XP(c * N + j), p1 = TG_XP(c * N + j + 1), p2 = TG_XP(c * N + j + 2), p3 = TG_XP(c * N + j + 3);
        I.k3[c] = p0 * (-1 / 6.0) + p1 * (1 / 2.0) + p2 * (-1 / 2.0) + p3 * (1 / 6.0);
        I.k2[c] = p0 * (1 / 2.0) + p1 * (-1.0) + p2 * (1 / 2.0);
        I.k1[c] = p0 * (-1 / 2.0) + p2 * (1 / 2.0);
    }
}

template <int D>
TG_HD double tg_dot(const double *a, const double *b)
{
    double s = 0;
#pragma unroll
    for (int c = 0; c < D; c++) s += a[c] * b[c];
    return s;
}

template <int D>
TG_HD double tg_norm(const double *a)
{
    return sqrt(tg_dot<D>(a, a));
}

// velocity / acceleration at time t on an interval of duration alpha
// (CC/src/DerivativeEvaluator.cpp:22-46, 83-128)
template <int D>
TG_HD void tg_velocity(const TgInterval<D> &I, double t, double al, double *v)
{
    const double T0 = 3 * t * t / (al * al * al), T1 = 2 * t / (al * al), T2 = 1 / al;
#pragma unroll
    for (int c = 0; c < D; c++) v[c] = I.k3[c] * T0 + I.k2[c] * T1 + I.k1[c] * T2;
}

template <int D>
TG_HD void tg_acceleration(const TgInterval<D> &I, double t, double al, double *a)
{
    const double T0 = 6 * t / (al * al * al), T1 = 2 / (al * al);
#pragma unroll
    for (int c = 0; c < D; c++) a[c] = I.k3[c] * T0 + I.k2[c] * T1;
}

// d v_c / d P_{c,l} and d a_c / d P_{c,l} at time t
TG_HD double tg_cv(int l, double t, double al)
{
    return TG_C3(l) * (3 * t * t / (al * al * al)) + TG_C2(l) * (2 * t / (al * al)) + TG_C1(l) / al;
}
TG_HD double tg_ca(int l, double t, double al)
{
    return TG_C3(l) * (6 * t / (al * al * al)) + TG_C2(l) * (2 / (al * al));
}

// gl[c*4+l] += dq/dv_c * dv_c/dP_{c,l} + dq/da_c * da_c/dP_{c,l}
template <int D>
TG_HD void tg_chain(double *gl, double scale, const double *dv, const double *da, double t, double al)
{
#pragma unroll
    for (int l = 0; l < 4; l++) {
        const double cv = tg_cv(l, t, al), ca = tg_ca(l, t, al);
#pragma unroll
        for (int c = 0; c < D; c++) gl[c * 4 + l] += scale * (dv[c] * cv + da[c] * ca);
    }
}

// ---- exact minimum speed on an interval, CC/src/DerivativeBounds.cpp:48-76, 110-123 ----
template <int D>
TG_FN void tg_min_velocity(const TgInterval<D> &I, double al, double &vmin, double &tmin)
{
    const double J00 = tg_dot<D>(I.k3, I.k3), J01 = tg_dot<D>(I.k3, I.k2), J11 = tg_dot<D>(I.k2, I.k2),
                 J20 = tg_dot<D>(I.k1, I.k3), J21 = tg_dot<D>(I.k1, I.k2);
    double r[3], v[D];
    tg_solve_cubic_eq(36 * J00, 12 * J01 + 24 * J01, 8 * J11 + 12 * J20, 4 * J21, r);
    tg_velocity<D>(I, 0.0, al, v);
    double best = tg_norm<D>(v), tb = 0;
    tg_velocity<D>(I, al, al, v);
    double s = tg_norm<D>(v);
    if (s < best) { best = s; tb = al; }
#pragma unroll
    for (int i = 0; i < 3; i++) {
        const double t = r[i] * al;
        if (t > 0 && t < al) {
            tg_velocity<D>(I, t, al, v);
            s = tg_norm<D>(v);
            if (s < best) { best = s; tb = t; }
        }
    }
    vmin = best; tmin = tb;
}

// gradient of the interval's min speed w.r.t. its 4 control points (gl[c*4+l] +=), envelope at tmin
template <int D>
TG_FN void tg_min_velocity_grad(const TgInterval<D> &I, double al, double vmin, double tmin, double scale, double *gl)
{
    if (!(vmin > 0)) return;
    double v[D], z[D];
    tg_velocity<D>(I, tmin, al, v);
#pragma unroll
    for (int c = 0; c < D; c++) { v[c] /= vmin; z[c] = 0; }
    tg_chain<D>(gl, scale, v, z, tmin, al);
}

// ---- |v x a| at time t, CC/src/CrossTermEvaluator.cpp:13-19, 75-92 ----
template <int D>
TG_HD double tg_cross_term(const TgInterval<D> &I, double t, double al)
{
    double v[D], a[D];
    tg_velocity<D>(I, t, al, v);
    tg_acceleration<D>(I, t, al, a);
    if (D == 2) return fabs(v[0] * a[1] - v[1] * a[0]);
    const double x = v[1] * a[D - 1] - v[D - 1] * a[1], y = v[D - 1] * a[0] - v[0] * a[D - 1], z = v[0] * a[1] - v[1] * a[0];
    return sqrt(x * x + y * y + z * z);
}

template <int D>
TG_HD void tg_cross3(const double *a, const double *b, double *o)
{
    if (D == 2) { o[0] = 0; o[1] = 0; o[2] = a[0] * b[1] - a[1] * b[0]; }
    else { o[0] = a[1] * b[D - 1] - a[D - 1] * b[1]; o[1] = a[D - 1] * b[0] - a[0] * b[D - 1]; o[2] = a[0] * b[1] - a[1] * b[0]; }
}

// ---- max |v x a| on an interval, CC/src/CrossTermBounds.cpp:168-200; cubic
// coefficients of d|v x a|^2/dtau from CC/src/CrossTermProperties.cpp:13-101:
// alpha^3 (v x a) = 6 U tau^2 + 6 V tau + 2 W, U = k2 x k3, V = k1 x k3, W = k1 x k2 ----
template <int D>
TG_FN void tg_max_cross_term(const TgInterval<D> &I, double al, double &cmax, double &tmax)
{
    double U[3], V[3], W[3], r[3];
    tg_cross3<D>(I.k2, I.k3, U); tg_cross3<D>(I.k1, I.k3, V); tg_cross3<D>(I.k1, I.k2, W);
    tg_solve_cubic_eq(72 * tg_dot<3>(U, U), 108 * tg_dot<3>(U, V), 36 * tg_dot<3>(V, V) + 24 * tg_dot<3>(U, W),
                      12 * tg_dot<3>(V, W), r);
    double best = tg_cross_term<D>(I, 0.0, al), tb = 0;
    double s = tg_cross_term<D>(I, al, al);
    if (s > best) { best = s; tb = al; }
#pragma unroll
    for (int i = 0; i < 3; i++) {
        const double t = r[i] * al;
        if (t > 0 && t < al) {
            s = tg_cross_term<D>(I, t, al);
            if (s > best) { best = s; tb = t; }
        }
    }
    cmax = best; tmax = tb;
}

// ---- conservative turning bound of one interval, CC/src/CrossTermBounds.cpp:64-152.
// kind: TG_TURN_CURVATURE (alpha forced to 1), ANGULAR_RATE, CENTRIPETAL.
// If gl != nullptr it receives d bound / d P (gl[c*4+l], overwritten); the alpha
// derivative is (p-2) bound / alpha by homogeneity (p = 2, 1, 0). ----
template <int D>
TG_FN double tg_interval_turn_bound(const TgInterval<D> &I, double al, int kind, double *gl)
{
    if (kind == TG_TURN_CURVATURE) al = 1.0;
    if (gl) {
#pragma unroll
        for (int q = 0; q < 4 * D; q++) gl[q] = 0;
    }
    double vmin, tv, cmax, tc;
    tg_min_velocity<D>(I, al, vmin, tv);
    tg_max_cross_term<D>(I, al, cmax, tc);
    double a0[D], a1[D];
    tg_acceleration<D>(I, 0.0, al, a0);
    tg_acceleration<D>(I, al, al, a1);
    const double n0 = tg_norm<D>(a0), n1 = tg_norm<D>(a1);
    const double amax = n1 > n0 ? n1 : n0;      // CC/src/DerivativeBounds.cpp:128-142
    const double ta = n1 > n0 ? al : 0.0;
    if (vmin <= 1.0e-8) {
        if (kind == TG_TURN_CENTRIPETAL) return 0;
        double at[D];
        tg_acceleration<D>(I, tv, al, at);
        return tg_norm<D>(at) <= 1.0e-8 ? 0 : DBL_MAX;
    }
    const int p = kind == TG_TURN_CURVATURE ? 2 : kind == TG_TURN_ANGULAR_RATE ? 1 : 0;
    double vp = 1;   // vmin^p
    #pragma unroll 1
    for (int q = 0; q < p; q++) vp *= vmin;
    const double b1 = amax / vp, b2 = cmax / (vp * vmin);
    const bool use2 = b2 < b1;
    if (gl) {
        double zero[D], dv[D], da[D];
#pragma unroll
        for (int c = 0; c < D; c++) zero[c] = 0;
        if (use2) {
            // d cmax
            double v[D], a[D], w[3];
            tg_velocity<D>(I, tc, al, v);
            tg_acceleration<D>(I, tc, al, a);
            tg_cross3<D>(v, a, w);
            if (cmax > 0) {
                if (D == 2) {
                    const double sg = w[2] < 0 ? -1.0 : 1.0;
                    dv[0] = sg * a[1]; dv[1] = -sg * a[0];
                    da[0] = -sg * v[1]; da[1] = sg * v[0];
                } else {
                    const double nx = w[0] / cmax, ny = w[1] / cmax, nz = w[2] / cmax;
                    // d|w|/dv = a x n ; d|w|/da = n x v
                    dv[0] = a[1] * nz - a[D - 1] * ny; dv[1] = a[D - 1] * nx - a[0] * nz; dv[D - 1] = a[0] * ny - a[1] * nx;
                    da[0] = ny * v[D - 1] - nz * v[1]; da[1] = nz * v[0] - nx * v[D - 1]; da[D - 1] = nx * v[1] - ny * v[0];
                }
                tg_chain<D>(gl, 1.0 / (vp * vmin), dv, da, tc, al);
            }
            tg_min_velocity_grad<D>(I, al, vmin, tv, -(p + 1) * b2 / vmin, gl);
        } else {
            if (amax > 0) {
                const double *am = n1 > n0 ? a1 : a0;
#pragma unroll
                for (int c = 0; c < D; c++) da[c] = am[c] / amax;
                tg_chain<D>(gl, 1.0 / vp, zero, da, ta, al);
            }
            if (p > 0) tg_min_velocity_grad<D>(I, al, vmin, tv, -p * b1 / vmin, gl);
        }
    }
    return use2 ? b2 : b1;
}

// ---------------------------------------------------------------------------
// B-spline -> MINVO, third order.  MV: CC/src/BsplineToMinvo.cpp:87-96 (obstacles).
// The SFC block uses the Python matrix whose end columns are the curve end
// points (TG/control_point_conversions/bspline_to_minvo.py:44-48).
// Q_k = sum_l P_l MV[l][k].
// ---------------------------------------------------------------------------
#define TG_MVA 0.18372189964688778830269864557208
#define TG_MVB 0.057009542139797595613306102386893
#define TG_MVC (-0.015455156825262485566573649098775)
#define TG_MVD (-0.0053387946850481119404479942697845)
#define TG_MVE 0.7017652268843997637057156686535
#define TG_MVF 0.66657381574108923111064205020873
#define TG_MVG 0.2918717989443756838876956809183
#define TG_MVH 0.11985166815376058497710386445935

TG_HD double tg_minvo(int l, int k)
{
    // rows l = 0..3, columns k = 0..3; row 3-l is row l reversed
    const int ll = l < 2 ? l : 3 - l, kk = l < 2 ? k : 3 - k;
    if (ll == 0) return kk == 0 ? TG_MVA : kk == 1 ? TG_MVB : kk == 2 ? TG_MVC : TG_MVD;
    return kk == 0 ? TG_MVE : kk == 1 ? TG_MVF : kk == 2 ? TG_MVG : TG_MVH;
}

TG_HD double tg_minvo_py(int l, int k)
{
    if (k == 0) return l == 0 ? 1.0 / 6.0 : l == 1 ? 2.0 / 3.0 : l == 2 ? 1.0 / 6.0 : 0.0;
    if (k == 3) return l == 0 ? 0.0 : l == 1 ? 1.0 / 6.0 : l == 2 ? 2.0 / 3.0 : 1.0 / 6.0;
    return tg_minvo(l, k);
}

// the same 16 numbers as a table, [l][k] (one load instead of a tree of selects: the QP stage regenerates corridor
// normals from them in several places and its instruction footprint is what its warps wait on)
#define TG_MV_ROW(l) {tg_minvo_py_c(l, 0), tg_minvo_py_c(l, 1), tg_minvo_py_c(l, 2), tg_minvo_py_c(l, 3)}
#define tg_minvo_py_c(l, k) ((k) == 0 ? ((l) == 0 ? 1.0 / 6.0 : (l) == 1 ? 2.0 / 3.0 : (l) == 2 ? 1.0 / 6.0 : 0.0) : \
                             (k) == 3 ? ((l) == 0 ? 0.0 : (l) == 1 ? 1.0 / 6.0 : (l) == 2 ? 2.0 / 3.0 : 1.0 / 6.0) : \
                             (((l) < 2 ? (l) : 3 - (l)) == 0 ? (((l) < 2 ? (k) : 3 - (k)) == 1 ? TG_MVB : TG_MVC) : (((l) < 2 ? (k) : 3 - (k)) == 1 ? TG_MVF : TG_MVG)))
#ifdef __CUDACC__
static __device__ const double tg_minvo_py_dev[4][4] = {TG_MV_ROW(0), TG_MV_ROW(1), TG_MV_ROW(2), TG_MV_ROW(3)};
#endif
TG_HD double tg_minvo_py_t(int l, int k)
{
#ifdef __CUDA_ARCH__
    return tg_minvo_py_dev[l][k];
#else
    return tg_minvo_py(l, k);
#endif
}

// ---- signed clearance of interval j's MINVO hull to a sphere,
// CC/src/SphereCollisionEvaluator.cpp:88-154 (rotation written as the unit
// vector u = first row of R, SURVEY.md A.6).  gl (optional): d dist / d P. ----
template <int D>
TG_FN double tg_hull_distance(const double *x, int N, int j, const double *center, double radius, double *gl,
                              int pi = -1, double pv = 0)
{
    double q[D][4], w[D];
#pragma unroll
    for (int c = 0; c < D; c++) {
        const double p0 = TG_XP(c * N + j), p1 = TG_XP(c * N + j + 1), p2 = TG_XP(c * N + j + 2), p3 = TG_XP(c * N + j + 3);
#pragma unroll
        for (int k = 0; k < 4; k++)
            q[c][k] = p0 * tg_minvo(0, k) + p1 * tg_minvo(1, k) + p2 * tg_minvo(2, k) + p3 * tg_minvo(3, k);
        w[c] = (q[c][0] + q[c][1] + q[c][2] + q[c][3]) / 4 - center[c];
    }
    const double wn = tg_norm<D>(w);
    double u[D];
    if (wn == 0) {
#pragma unroll
        for (int c = 0; c < D; c++) u[c] = c == 0 ? 1.0 : 0.0;
    } else {
#pragma unroll
        for (int c = 0; c < D; c++) u[c] = w[c] / wn;
    }
    double minx = DBL_MAX;
    int ks = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        double s = 0;
#pragma unroll
        for (int c = 0; c < D; c++) s += u[c] * q[c][k];
        if (s < minx) { minx = s; ks = k; }
    }
    const double cx = tg_dot<D>(u, center);
    if (gl) {
        // d/dQ_l = u delta_{l,ks} + (I - u u^T)(Q_ks - c) / (4 |w|)
        double h[D], e[D];
#pragma unroll
        for (int c = 0; c < D; c++) e[c] = q[c][ks] - center[c];
        const double ue = tg_dot<D>(u, e);
#pragma unroll
        for (int c = 0; c < D; c++) h[c] = wn == 0 ? 0.0 : (e[c] - ue * u[c]) / (4 * wn);
#pragma unroll
        for (int l = 0; l < 4; l++) {
            const double rowsum = tg_minvo(l, 0) + tg_minvo(l, 1) + tg_minvo(l, 2) + tg_minvo(l, 3);
            const double mk = tg_minvo(l, ks);
#pragma unroll
            for (int c = 0; c < D; c++) gl[c * 4 + l] = mk * u[c] + rowsum * h[c];
        }
    }
    return minx - (cx + radius);
}

// ---------------------------------------------------------------------------
// objective and gradient, TG/objectives/objective_functions.py:6-62
// ---------------------------------------------------------------------------
TG_HD double tg_stencil(int k, int t)
{
    if (k == 1) return t == 0 ? 1.0 : -1.0;
    if (k == 2) return t == 1 ? -2.0 : 1.0;
    return t == 0 ? -1.0 : t == 1 ? 3.0 : t == 2 ? -3.0 : 1.0;
}

TG_HD double tg_diff(const double *row, int k, int j)
{
    if (k == 1) return row[j] - row[j + 1];
    if (k == 2) return row[j + 2] - 2 * row[j + 1] + row[j];
    return row[j + 3] - 3 * row[j + 2] + 3 * row[j + 1] - row[j];
}

// returns f on every lane; g (n entries, optional) is complete after TG_SYNC()
TG_EVAL_FN double tg_objective(const TgLayout &L, const int *sp, const double *x, double *g)
{
    const int obj = sp[TG_SP_OBJECTIVE], d = L.d, N = L.N, lane = TG_LANE();
    const double al = x[L.ia];
    const int k = (obj == TG_OBJ_DIST || obj == TG_OBJ_DIST_TIME || obj == TG_OBJ_TIME_VEL_PENALTY) ? 1
                : (obj == TG_OBJ_VEL || obj == TG_OBJ_VEL_TIME) ? 2 : (obj == TG_OBJ_ACC || obj == TG_OBJ_ACC_TIME) ? 3 : 0;
    double S = 0;
    if (k) {
        const int nd = N - k;
        #pragma unroll 1
        for (int q = lane; q < d * nd; q += TG_NL) {
            const int c = q / nd, j = q - c * nd;
            const double dd = tg_diff(x + c * N, k, j);
            S += dd * dd;
        }
        S = tg_wsum(S);
    }
    double wS, f, dfa;   // f = wS * S + (alpha part)
    switch (obj) {
    case TG_OBJ_TIME: wS = 0; f = al * al; dfa = 2 * al; break;
    case TG_OBJ_DIST: case TG_OBJ_VEL: case TG_OBJ_ACC: wS = 1; f = S; dfa = 0; break;
    case TG_OBJ_DIST_TIME: case TG_OBJ_VEL_TIME: case TG_OBJ_ACC_TIME: wS = al; f = S * al; dfa = S; break;
    default: wS = -1; f = 100 * al * al - S; dfa = 200 * al; break;
    }
    if (g) {
        #pragma unroll 1
        for (int q = lane; q < L.n; q += TG_NL) {
            double v = 0;
            if (q < d * N) {
                if (k) {
                    const int c = q / N, i = q - c * N;
                    double s = 0;
                    #pragma unroll 1
                    for (int t = 0; t <= k; t++) {
                        const int j = i - t;
                        if (j >= 0 && j < N - k) s += tg_stencil(k, t) * tg_diff(x + c * N, k, j);
                    }
                    v = 2 * wS * s;
                }
            } else if (q == L.ia) v = dfa;
            g[q] = v;
        }
    }
    return f;
}

// ---------------------------------------------------------------------------
// constraint blocks
// ---------------------------------------------------------------------------

// terminal location rows (linear): CF/waypoint_constraints.py:10-71, 122-147
TG_FN void tg_rows_location(const TgLayout &L, const int *sp, const double *par, const double *x, double *c)
{
    const int d = L.d, N = L.N, lane = TG_LANE();
    #pragma unroll 1
    for (int q = lane; q < L.n_start + L.n_end; q += TG_NL) {
        const bool start = q < L.n_start;
        const int r = start ? q : q - L.n_start;
        const int kind = start ? sp[TG_SP_START_KIND] : sp[TG_SP_END_KIND];
        const double *loc = par + (start ? L.p_start_loc : L.p_end_loc);
        double v;
        if (kind == 1) {          // zero velocity: three control points pinned to the waypoint
            const int i = r / 3, l = r - 3 * i;
            v = x[start ? i * N + l : (i + 1) * N - 3 + l] - loc[i];
        } else {
            const double *p = x + (start ? r * N : (r + 1) * N - 3);
            v = p[0] / 6.0 + p[1] * (2.0 / 3.0) + p[2] / 6.0 - loc[r];
            if (!start && kind == 2) v -= (N - 3) * par[L.p_target_vel + r] * x[L.ia];
        }
        c[(start ? L.r_start : L.r_end) + r] = v;
    }
}

// constant Jacobian rows of the location blocks (called once per problem)
TG_FN void tg_jac_location(const TgLayout &L, const int *sp, const double *par, const TgJac &J)
{
    const int d = L.d, N = L.N, lane = TG_LANE();
    (void)d;
    #pragma unroll 1
    for (int q = lane; q < L.n_start + L.n_end; q += TG_NL) {
        const bool start = q < L.n_start;
        const int r = start ? q : q - L.n_start;
        const int kind = start ? sp[TG_SP_START_KIND] : sp[TG_SP_END_KIND];
        double *row = J.p + ((start ? L.r_start : L.r_end) + r) * J.rs;
        #pragma unroll 1
        for (int i = 0; i < L.n; i++) row[i * J.cs] = 0;
        if (kind == 1) {
            const int i = r / 3, l = r - 3 * i;
            row[(start ? i * N + l : (i + 1) * N - 3 + l) * J.cs] = 1.0;
        } else {
            const int b = start ? r * N : (r + 1) * N - 3;
            row[b * J.cs] = 1.0 / 6.0; row[(b + 1) * J.cs] = 2.0 / 3.0; row[(b + 2) * J.cs] = 1.0 / 6.0;
            if (!start && kind == 2) row[L.ia * J.cs] = -(N - 3) * par[L.p_target_vel + r];
        }
    }
}

// terminal derivative rows (nonlinear equalities): CF/waypoint_constraints.py:73-120, 205-245
TG_FN void tg_rows_terminal(const TgLayout &L, const int *sp, const double *par, const double *x, double *cv,
                            const TgJac *J)
{
    const int d = L.d, N = L.N, lane = TG_LANE();
    const double al = x[L.ia];
    #pragma unroll 1
    for (int side = 0; side < 2; side++) {
        const int dirk = sp[side ? TG_SP_END_DIR : TG_SP_START_DIR];
        const int velon = sp[side ? TG_SP_END_VEL : TG_SP_START_VEL], accon = sp[side ? TG_SP_END_ACC : TG_SP_START_ACC];
        const int nrows = side ? L.n_eder : L.n_sder, r0 = side ? L.r_eder : L.r_sder;
        #pragma unroll 1
        for (int q = lane; q < nrows; q += TG_NL) {
            int blk = q / d;
            const int c = q - blk * d;
            // block order: direction, velocity, acceleration (present ones only)
            int what;    // 0 dir 1 vel 2 acc
            if (dirk) { what = blk == 0 ? 0 : (blk == 1 && velon) ? 1 : 2; }
            else { what = (blk == 0 && velon) ? 1 : 2; }
            const int i0 = c * N + (side ? N - 3 : 0);      // first of the three end control points
            const double first = x[i0], mid = x[i0 + 1], last = x[i0 + 2];
            double *row = J ? tg_jrow(*J, L, r0 + q) : 0;
            const int cs = J ? J->cs : 0;
            double v;
            if (what == 0) {
                const int is = side ? L.is1 : L.is0;
                const double s = x[is];
                int ia_, ib_;   // direction ~ s (x[ib_] - x[ia_]) / 2
                if (dirk == 2) { ia_ = side ? c * N + N - 4 : c * N; ib_ = side ? c * N + N - 1 : c * N + 3; }
                else { ia_ = i0; ib_ = i0 + 2; }
                const double diff = x[ib_] - x[ia_];
                v = s * diff / 2 - par[(side ? L.p_edir : L.p_sdir) + c];
                if (row) { row[ib_ * cs] = s / 2; row[ia_ * cs] = -s / 2; row[is * cs] = diff / 2; }
            } else if (what == 1) {
                v = (last - first) / (2 * al) - par[(side ? L.p_evel : L.p_svel) + c];
                if (row) {
                    row[(i0 + 2) * cs] = 1 / (2 * al); row[i0 * cs] = -1 / (2 * al);
                    row[L.ia * cs] = -(last - first) / (2 * al * al);
                }
            } else {
                v = (first - 2 * mid + last) / (al * al) - par[(side ? L.p_eacc : L.p_sacc) + c];
                if (row) {
                    row[i0 * cs] = 1 / (al * al); row[(i0 + 1) * cs] = -2 / (al * al); row[(i0 + 2) * cs] = 1 / (al * al);
                    row[L.ia * cs] = -2 * (first - 2 * mid + last) / (al * al * al);
                }
            }
            cv[r0 + q] = v;
        }
    }
}

// intermediate waypoint rows: CF/waypoint_constraints.py:248-295 (interval = int(tau))
TG_FN void tg_rows_intermediate(const TgLayout &L, const int *sp, const double *par, const double *x, double *cv,
                                const TgJac *J)
{
    const int d = L.d, N = L.N, niw = L.niw, lane = TG_LANE();
    const double al = x[L.ia];
    const int nitems = d * niw * (sp[TG_SP_IW_VEL] ? 2 : 1);
    #pragma unroll 1
    for (int q = lane; q < nitems; q += TG_NL) {
        const int vel = q >= d * niw;
        const int qq = vel ? q - d * niw : q;
        const int c = qq / niw, i = qq - c * niw;       // rows are (d, niw).flatten()
        const double tau = x[L.it0 + i];
        int k = (int)tau;
        const double u = tau - k;
        const int r = (vel ? L.r_iwv : L.r_iwl) + qq;
        double *row = J ? tg_jrow(*J, L, r) : 0;
        const int cs = J ? J->cs : 0;
        const double *p = x + c * N + k;
        double v;
        if (k >= N - 3) {
            // tau == N-3: the reference slices 3 control points and evaluates an order-2 spline at u = 0
            // (CF/waypoint_constraints.py:261, TG/matrix_evaluation.py:184, SURVEY.md A.4)
            k = N - 3; p = x + c * N + k;
            if (!vel) {
                v = 0.5 * p[0] + 0.5 * p[1] - par[L.p_iwl + qq];
                if (row) { row[(c * N + k) * cs] = 0.5; row[(c * N + k + 1) * cs] = 0.5; row[(L.it0 + i) * cs] = p[1] - p[0]; }
            } else {
                const double vv = (p[1] - p[0]) / al;
                v = vv - par[L.p_iwv + qq];
                if (row) {
                    row[(c * N + k) * cs] = -1 / al; row[(c * N + k + 1) * cs] = 1 / al;
                    row[(L.it0 + i) * cs] = (p[0] - 2 * p[1] + p[2]) / al; row[L.ia * cs] = -vv / al;
                }
            }
            cv[r] = v;
            continue;
        }
        if (!vel) {
            double s = 0, ds = 0;
#pragma unroll
            for (int l = 0; l < 4; l++) {
                const double k0l = l == 0 ? 1.0 / 6.0 : l == 1 ? 2.0 / 3.0 : l == 2 ? 1.0 / 6.0 : 0.0;
                const double b = ((TG_C3(l) * u + TG_C2(l)) * u + TG_C1(l)) * u + k0l;
                const double db = (3 * TG_C3(l) * u + 2 * TG_C2(l)) * u + TG_C1(l);
                s += p[l] * b; ds += p[l] * db;
                if (row) row[(c * N + k + l) * cs] = b;
            }
            v = s - par[L.p_iwl + qq];
            if (row) row[(L.it0 + i) * cs] = ds;
        } else {
            double s = 0, ds = 0;
#pragma unroll
            for (int l = 0; l < 4; l++) {
                const double b = ((3 * TG_C3(l) * u + 2 * TG_C2(l)) * u + TG_C1(l)) / al;
                const double db = (6 * TG_C3(l) * u + 2 * TG_C2(l)) / al;
                s += p[l] * b; ds += p[l] * db;
                if (row) row[(c * N + k + l) * cs] = b;
            }
            v = s - par[L.p_iwv + qq];
            if (row) { row[(L.it0 + i) * cs] = ds; row[L.ia * cs] = -s / al; }
        }
        cv[r] = v;
    }
}

// Bezier velocity point b_q of the spline (q = 0 .. 2 nint):
// TG/control_point_conversions/bspline_to_bezier.py:23-45 applied to V_j = (P_{j+1}-P_j)/alpha.
// b_q = sum_t wq[t] P_{i0+t} / alpha.
TG_HD void tg_bezier_vel_weights(int q, int &i0, double wq[3])
{
    const int i = q >> 1;
    i0 = i;
    if (q & 1) { i0 = i + 1; wq[0] = -1.0; wq[1] = 1.0; wq[2] = 0.0; }       // V_{i+1}
    else { wq[0] = -0.5; wq[1] = 0.0; wq[2] = 0.5; }                          // (V_i + V_{i+1}) / 2
}

// derivative-bound rows: CF/derivative_constraints.py:17-121.  Each row is max/min over
// points; rows are emitted as (limit - value) >= 0.
template <int D>
TG_FN void tg_rows_derivative(const TgLayout &L, const int *sp, const double *par, const double *x, double *cv,
                              const TgJac *J)
{
    const int N = L.N, nint = L.nint, lane = TG_LANE();
    const double al = x[L.ia];
    int r = L.r_db;
    const int cs = J ? J->cs : 0;
    if (sp[TG_SP_DB_MINV]) {
        // min speed over the spline: CC/src/DerivativeBounds.cpp:12-27
        double best = DBL_MAX, tbest = 0; int jb = 0x7fffffff;
        #pragma unroll 1
        for (int j = lane; j < nint; j += TG_NL) {
            TgInterval<D> I; double v, t;
            tg_load_interval<D>(x, N, j, I);
            tg_min_velocity<D>(I, al, v, t);
            if (v < best) { best = v; tbest = t; jb = j; }
        }
        double bv = best; int bj = jb;
        tg_wargmin(bv, bj);
        if (lane == 0) cv[r] = bv - par[L.p_minv];
        if (J && jb == bj && bj != 0x7fffffff) {
            double gl[4 * D];
#pragma unroll
            for (int q = 0; q < 4 * D; q++) gl[q] = 0;
            TgInterval<D> I;
            tg_load_interval<D>(x, N, bj, I);
            tg_min_velocity_grad<D>(I, al, best, tbest, 1.0, gl);
            double *row = tg_jrow(*J, L, r);
#pragma unroll
            for (int c = 0; c < D; c++)
#pragma unroll
                for (int l = 0; l < 4; l++) row[(c * N + bj + l) * cs] = gl[c * 4 + l];
            row[L.ia * cs] = -best / al;
        }
        r++;
    }
    if (sp[TG_SP_DB_MAXV]) {
        const int npt = 2 * nint + 1;
        // which = 0: max |b|, 1: -min b_z (upward), 2: max |b_xy| (horizontal)
        #pragma unroll 1
        for (int which = 0; which < 3; which++) {
            if (which == 1 && !sp[TG_SP_DB_UP]) continue;
            if (which == 2 && !sp[TG_SP_DB_HORIZ]) continue;
            const double lim = par[which == 0 ? L.p_maxv : which == 1 ? L.p_up : L.p_horiz];
            // in 2-D these rows are allocated but never written and the later rows move up
            // (CF/derivative_constraints.py:38-43 vs :71-76); the unwritten tail is zeroed below
            if (which > 0 && D == 2) continue;
            double best = -DBL_MAX; int qb = 0x7fffffff;
            #pragma unroll 1
            for (int q = lane; q < npt; q += TG_NL) {
                int i0; double wq[3], b[D];
                tg_bezier_vel_weights(q, i0, wq);
#pragma unroll
                for (int c = 0; c < D; c++)
                    b[c] = (wq[0] * x[c * N + i0] + wq[1] * x[c * N + i0 + 1] + wq[2] * x[c * N + i0 + 2]) / al;
                double s;
                if (which == 0) s = tg_norm<D>(b);
                else if (which == 1) s = -b[D - 1];
                else s = sqrt(b[0] * b[0] + b[1] * b[1]);
                if (s > best) { best = s; qb = q; }
            }
            double bv = best; int bq = qb;
            tg_wargmax(bv, bq);
            if (lane == 0) cv[r] = lim - bv;
            if (J && qb == bq) {
                int i0; double wq[3], b[D];
                tg_bezier_vel_weights(bq, i0, wq);
#pragma unroll
                for (int c = 0; c < D; c++)
                    b[c] = (wq[0] * x[c * N + i0] + wq[1] * x[c * N + i0 + 1] + wq[2] * x[c * N + i0 + 2]) / al;
                double *row = tg_jrow(*J, L, r);
                double da = 0;
#pragma unroll
                for (int c = 0; c < D; c++) {
                    double dsdb;   // d s / d b_c
                    if (which == 0) dsdb = bv > 0 ? b[c] / bv : 0.0;
                    else if (which == 1) dsdb = c == D - 1 ? -1.0 : 0.0;
                    else dsdb = (c < 2 && bv > 0) ? b[c] / bv : 0.0;
                    #pragma unroll 1
                    for (int t = 0; t < 3; t++)
                        if (wq[t] != 0) row[(c * N + i0 + t) * cs] = -dsdb * wq[t] / al;
                    da += dsdb * b[c];
                }
                row[L.ia * cs] = da / al;     // -(d s/d alpha) = +s/alpha
            }
            r++;
        }
    }
    // acceleration control points A_j = (P_j - 2 P_{j+1} + P_{j+2}) / alpha^2 (minus gravity in 3-D), jerk J_j = D3_j / alpha^3
    #pragma unroll 1
    for (int which = 0; which < 2; which++) {
        if (!sp[which == 0 ? TG_SP_DB_MAXA : TG_SP_DB_JERK]) continue;
        const int npt = which == 0 ? N - 2 : N - 3;
        const double grav = (which == 0 && sp[TG_SP_DB_GRAV] && D == 3) ? par[L.p_grav] : 0.0;
        const double sc = which == 0 ? 1 / (al * al) : 1 / (al * al * al);
        double best = -DBL_MAX; int qb = 0x7fffffff;
        #pragma unroll 1
        for (int q = lane; q < npt; q += TG_NL) {
            double b[D];
#pragma unroll
            for (int c = 0; c < D; c++) b[c] = tg_diff(x + c * N, which == 0 ? 2 : 3, q) * sc;
            b[D - 1] -= grav;
            const double s = tg_norm<D>(b);
            if (s > best) { best = s; qb = q; }
        }
        double bv = best; int bq = qb;
        tg_wargmax(bv, bq);
        if (lane == 0) cv[r] = par[which == 0 ? L.p_maxa : L.p_jerk] - bv;
        if (J && qb == bq) {
            double b[D], raw[D];
#pragma unroll
            for (int c = 0; c < D; c++) { raw[c] = tg_diff(x + c * N, which == 0 ? 2 : 3, bq) * sc; b[c] = raw[c]; }
            b[D - 1] -= grav;
            double *row = tg_jrow(*J, L, r);
            double da = 0;
            const int k = which == 0 ? 2 : 3;
#pragma unroll
            for (int c = 0; c < D; c++) {
                const double dsdb = bv > 0 ? b[c] / bv : 0.0;
                #pragma unroll 1
                for (int t = 0; t <= k; t++) {
                    // tg_diff order 2: +P_j -2P_{j+1} +P_{j+2}; order 3: -P_j +3P_{j+1} -3P_{j+2} +P_{j+3}
                    const double st = k == 2 ? (t == 1 ? -2.0 : 1.0) : tg_stencil(3, t);
                    row[(c * N + bq + t) * cs] = -dsdb * st * sc;
                }
                da += dsdb * raw[c];
            }
            row[L.ia * cs] = k * da / al;
        }
        r++;
    }
    #pragma unroll 1
    for (int q = r + lane; q < L.r_db + L.n_db; q += TG_NL) cv[q] = -0.0;
}

// tangential acceleration rows: CF/derivative_constraints.py:124-241
template <int D>
TG_FN void tg_rows_tangential(const TgLayout &L, const int *sp, const double *par, const double *x, double *cv,
                              const TgJac *J)
{
    (void)sp;
    const int N = L.N, nint = L.nint, lane = TG_LANE();
    const double al = x[L.ia];
    const double lo_lim = par[L.p_tanmin], hi_lim = par[L.p_tanmax];
    const int cs = J ? J->cs : 0;
    #pragma unroll 1
    for (int j = lane; j < nint; j += TG_NL) {
        TgInterval<D> I;
        tg_load_interval<D>(x, N, j, I);
        // d(a.v)/dtau ~ c2 tau^2 + c1 tau + c0  (:186-229)
        const double c2 = 54 * tg_dot<D>(I.k3, I.k3), c1 = 36 * tg_dot<D>(I.k2, I.k3),
                     c0 = 4 * tg_dot<D>(I.k2, I.k2) + 6 * tg_dot<D>(I.k1, I.k3);
        double roots[2];
        const double disc = c1 * c1 - 4 * c2 * c0;       // :231-241 (division by zero -> inf / nan as numpy does)
        if (disc == 0) { roots[0] = -c1 / (2 * c2); roots[1] = INFINITY; }
        else if (disc < 0) { roots[0] = INFINITY; roots[1] = INFINITY; }
        else { const double sq = sqrt(disc); roots[0] = (-c1 + sq) / (2 * c2); roots[1] = (-c1 - sq) / (2 * c2); }
        double v[D], a[D];
        tg_velocity<D>(I, 0.0, al, v); tg_acceleration<D>(I, 0.0, al, a);
        double hi = tg_dot<D>(a, v), lo = hi, thi = 0, tlo = 0;
        #pragma unroll 1
        for (int q = 0; q < 3; q++) {
            const double t = q < 2 ? roots[q] * al : al;
            if (t < 0 || t > al) continue;
            tg_velocity<D>(I, t, al, v); tg_acceleration<D>(I, t, al, a);
            const double s = tg_dot<D>(a, v);
            if (s > hi) { hi = s; thi = t; }
            if (s < lo) { lo = s; tlo = t; }
        }
        double vmin, tv;
        tg_min_velocity<D>(I, al, vmin, tv);
        const double ymax = hi / vmin, ymin = lo / vmin;
        cv[L.r_tanl + j] = ymax - lo_lim;
        cv[L.r_tanl + nint + j] = ymin - lo_lim;
        cv[L.r_tanu + j] = hi_lim - ymax;
        cv[L.r_tanu + nint + j] = hi_lim - ymin;
        if (J) {
            #pragma unroll 1
            for (int e = 0; e < 2; e++) {
                const double s = e ? lo : hi, t = e ? tlo : thi;
                double gl[4 * D];
#pragma unroll
                for (int q = 0; q < 4 * D; q++) gl[q] = 0;
                tg_velocity<D>(I, t, al, v); tg_acceleration<D>(I, t, al, a);
                tg_chain<D>(gl, 1 / vmin, a, v, t, al);                        // d(a.v) = a.dv + v.da
                tg_min_velocity_grad<D>(I, al, vmin, tv, -s / (vmin * vmin), gl);
                const double dal = -2 * (s / vmin) / al;                       // (a.v) ~ alpha^-3, vmin ~ alpha^-1
                double *rl = tg_jrow(*J, L, L.r_tanl + e * nint + j), *ru = tg_jrow(*J, L, L.r_tanu + e * nint + j);
#pragma unroll
                for (int c = 0; c < D; c++)
#pragma unroll
                    for (int l = 0; l < 4; l++) {
                        rl[(c * N + j + l) * cs] = gl[c * 4 + l];
                        ru[(c * N + j + l) * cs] = -gl[c * 4 + l];
                    }
                rl[L.ia * cs] = dal; ru[L.ia * cs] = -dal;
            }
        }
    }
}

// turning row: CF/turning_constraints.py:49-121 -> CC/src/CrossTermBounds.cpp:13-61
template <int D>
TG_FN void tg_rows_turning(const TgLayout &L, const int *sp, const double *par, const double *x, double *cv,
                           const TgJac *J)
{
    const int N = L.N, lane = TG_LANE(), kind = sp[TG_SP_TURN];
    const double al = x[L.ia];
    const int first = L.turn_first, nint = L.turn_ncp - 3;
    double best = 0; int jb = 0x7fffffff;
    double gbest[4 * D], gl[4 * D];
    #pragma unroll 1
    for (int j = lane; j < nint; j += TG_NL) {
        TgInterval<D> I;
        tg_load_interval<D>(x, N, first + j, I);
        const double b = tg_interval_turn_bound<D>(I, al, kind, J ? gl : 0);
        if (b > best) {
            best = b; jb = j;
            if (J) {
#pragma unroll
                for (int q = 0; q < 4 * D; q++) gbest[q] = gl[q];
            }
        }
    }
    double bv = best; int bj = jb;
    tg_wargmax(bv, bj);
    const double scale = kind == TG_TURN_CURVATURE ? 100.0 : 1.0;       // CF/turning_constraints.py:56
    if (lane == 0) cv[L.r_turn] = -((bv - par[L.p_turn]) * scale);
    if (J && jb == bj && bj != 0x7fffffff && bv < DBL_MAX) {
        double *row = tg_jrow(*J, L, L.r_turn);
        const int cs = J->cs;
#pragma unroll
        for (int c = 0; c < D; c++)
#pragma unroll
            for (int l = 0; l < 4; l++) row[(c * N + first + bj + l) * cs] = -scale * gbest[c * 4 + l];
        const int p = kind == TG_TURN_CURVATURE ? 2 : kind == TG_TURN_ANGULAR_RATE ? 1 : 0;
        if (p != 2) row[L.ia * cs] = -scale * (p - 2) * bv / al;
    }
}

// SFC rows (linear): CF/sfc_constraints.py:7-77.  Row (rr, idx = 4 j + k) of each block.
template <int D>
TG_FN void tg_rows_sfc(const TgLayout &L, const int *sp, const double *par, const double *x, double *cv)
{
    const int N = L.N, nint = L.nint, lane = TG_LANE(), npts = 4 * nint;
    #pragma unroll 1
    for (int q = lane; q < npts; q += TG_NL) {
        const int j = q >> 2, k = q & 3;
        const double *cor = par + L.p_sfc + tg_corridor_of_interval(sp, j) * tg_sfc_stride(D);
        double Q[D];
#pragma unroll
        for (int c = 0; c < D; c++) {
            const double *p = x + c * N + j;
            Q[c] = p[0] * tg_minvo_py(0, k) + p[1] * tg_minvo_py(1, k) + p[2] * tg_minvo_py(2, k) + p[3] * tg_minvo_py(3, k);
        }
#pragma unroll
        for (int rr = 0; rr < D; rr++) {
            double s = 0;
#pragma unroll
            for (int c = 0; c < D; c++) s += cor[rr * D + c] * Q[c];
            cv[L.r_sfcl + rr * npts + q] = s - cor[D * D + rr];
            cv[L.r_sfcu + rr * npts + q] = cor[D * D + D + rr] - s;
        }
    }
}

template <int D>
TG_FN void tg_jac_sfc(const TgLayout &L, const int *sp, const double *par, const TgJac &J)
{
    const int N = L.N, nint = L.nint, lane = TG_LANE(), npts = 4 * nint;
    #pragma unroll 1
    for (int q = lane; q < npts * D; q += TG_NL) {
        const int rr = q / npts, idx = q - rr * npts;
        const int j = idx >> 2, k = idx & 3;
        const double *cor = par + L.p_sfc + tg_corridor_of_interval(sp, j) * tg_sfc_stride(D);
        double *rl = J.p + (L.r_sfcl + q) * J.rs, *ru = J.p + (L.r_sfcu + q) * J.rs;
        #pragma unroll 1
        for (int i = 0; i < L.n; i++) { rl[i * J.cs] = 0; ru[i * J.cs] = 0; }
#pragma unroll
        for (int c = 0; c < D; c++)
#pragma unroll
            for (int l = 0; l < 4; l++) {
                const double v = cor[rr * D + c] * tg_minvo_py(l, k);
                rl[(c * N + j + l) * J.cs] = v;
                ru[(c * N + j + l) * J.cs] = -v;
            }
    }
}

// obstacle rows: CF/obstacle_constraints.py:93-113 -> CC/src/SphereCollisionEvaluator.cpp:13-45.
// scratch: K * nint doubles readable by every lane.
template <int D>
TG_FN void tg_rows_obstacles(const TgLayout &L, const int *sp, const double *par, const double *x, double *cv,
                             const TgJac *J, double *scratch)
{
    (void)sp;
    const int N = L.N, nint = L.nint, K = L.n_obs, lane = TG_LANE();
    #pragma unroll 1
    for (int q = lane; q < K * nint; q += TG_NL) {
        const int i = q / nint, j = q - i * nint;
        double ctr[D];
#pragma unroll
        for (int c = 0; c < D; c++) ctr[c] = par[L.p_obs_c + c * K + i];
        scratch[q] = tg_hull_distance<D>(x, N, j, ctr, par[L.p_obs_r + i], 0);
    }
    TG_SYNC();
    #pragma unroll 1
    for (int i = lane; i < K; i += TG_NL) {
        double best = DBL_MAX; int jb = 0;
        #pragma unroll 1
        for (int j = 0; j < nint; j++)
            if (best > scratch[i * nint + j]) { best = scratch[i * nint + j]; jb = j; }
        cv[L.r_obs + i] = best;
        if (J) {
            double ctr[D], gl[4 * D];
#pragma unroll
            for (int c = 0; c < D; c++) ctr[c] = par[L.p_obs_c + c * K + i];
            tg_hull_distance<D>(x, N, jb, ctr, par[L.p_obs_r + i], gl);
            double *row = tg_jrow_hi(*J, L, L.r_obs + i);
            const int cs = J->cs;
#pragma unroll
            for (int c = 0; c < D; c++)
#pragma unroll
                for (int l = 0; l < 4; l++) row[(c * N + jb + l) * cs] = gl[c * 4 + l];
        }
    }
    TG_SYNC();
}

// per-problem scratch of the evaluators: obstacle x interval distances, and for the item-parallel finite-difference
// sweeps (tg_fd_turning / tg_fd_obstacles) 4 perturbed values per control-point variable + 2 per interval
TG_HD int tg_scratch_doubles(const TgLayout &L) { return (L.n_obs * L.nint > 0 ? L.n_obs * L.nint : 1) + 4 * L.d * L.N + 2 * L.nint + 2; }

// shared memory of one problem in the evaluation kernel (tg_kernels_eval.inc): variables, parameters, the evaluators'
// scratch and -- only when the caller does not ask for the constraint values -- a sink for them.  (The evaluators only
// WRITE constraint rows, so with `c` given they write straight to global memory: the corridor rows, most of C4's 209,
// leave the lanes as contiguous runs.)
TG_HD int tg_eval_group_doubles(const TgLayout &L, bool sink_c)
{
    return L.n + L.P + (sink_c ? L.m : 0) + tg_scratch_doubles(L) + 4;
}

// zero every nonlinear Jacobian row (they are rewritten sparsely on each evaluation)
TG_FN void tg_zero_nonlinear_rows(const TgLayout &L, const TgJac &J)
{
    const int lane = TG_LANE();
    #pragma unroll 1
    for (int r = 0; r < L.m; r++) {
        if (tg_nlrow(L, r) < 0) continue;
        double *row = r >= L.r_obs ? tg_jrow_hi(J, L, r) : tg_jrow(J, L, r);
        #pragma unroll 1
        for (int i = lane; i < L.n; i += TG_NL) row[i * J.cs] = 0;
    }
    TG_SYNC();
}

// all constraint values (m) and, if J, the nonlinear Jacobian rows.  skip: blocks to leave untouched -- the solver's
// finite-difference sweeps need neither the linear rows (terminal locations, corridors) nor the blocks that have
// their own item-parallel sweep.
#define TG_SKIP_LINEAR 1
#define TG_SKIP_TURNING 2
#define TG_SKIP_OBSTACLES 4
template <int D>
TG_EVAL_FN void tg_constraints_d(const TgLayout &L, const int *sp, const double *par, const double *x, double *cv,
                            const TgJac *J, double *scratch, int skip = 0)
{
    const bool nl_only = (skip & TG_SKIP_LINEAR) != 0;
    if (J) tg_zero_nonlinear_rows(L, *J);
    if (!nl_only) tg_rows_location(L, sp, par, x, cv);
    if (L.n_sder + L.n_eder) tg_rows_terminal(L, sp, par, x, cv, J);
    if (L.niw) tg_rows_intermediate(L, sp, par, x, cv, J);
    if (L.n_db) tg_rows_derivative<D>(L, sp, par, x, cv, J);
    if (L.n_tan) tg_rows_tangential<D>(L, sp, par, x, cv, J);
    if (L.n_turn && !(skip & TG_SKIP_TURNING)) tg_rows_turning<D>(L, sp, par, x, cv, J);
    if (L.n_sfc && !nl_only) tg_rows_sfc<D>(L, sp, par, x, cv);
    if (L.n_obs && !(skip & TG_SKIP_OBSTACLES)) tg_rows_obstacles<D>(L, sp, par, x, cv, J, scratch);
    TG_SYNC();
}

// ---------------------------------------------------------------------------
// Item-parallel forward differences of the two heavy blocks, as scipy forms them for the reference
// (approx_derivative '2-point', abs_step = TG_FD_STEP, bounds):  A[i * lda + row] = (c(x + h_i e_i) - c(x)) / dx_i.
// A control-point variable only moves the (at most 4) intervals that contain it, so instead of n full
// re-evaluations the lanes work through the (interval, local control point, coordinate) items -- each one interval
// evaluation with the perturbation applied on load -- and the max / min over intervals is then taken per variable
// over perturbed values inside its window and base values outside.  Same numbers as n full evaluations.
// ---------------------------------------------------------------------------
#define TG_FD_STEP 1.4901161193847656e-08     // scipy/optimize/_slsqp_py.py:34

// bound-aware forward step (scipy/optimize/_numdiff.py: the step is flipped when x + h leaves [lo, hi] and the
// other side has room)
TG_HD double tg_fd_step(double xi, double lo, double hi)
{
    double h = TG_FD_STEP;
    const double xt = xi + h;
    if (xt < lo || xt > hi) {
        const double ld = xi - lo, ud = hi - xi;
        if (fabs(h) <= fmax(ld, ud)) h = -h;
        else h = ud >= ld ? ud : -ld;
    }
    return h;
}

// scr: 4 d N + 2 nint doubles
template <int D>
TG_EVAL_FN void tg_fd_turning(const TgLayout &L, const int *sp, const double *par, const double *x, const double *xl,
                         const double *xu, double c0, double *A, int lda, double *scr)
{
    const int N = L.N, lane = TG_LANE(), kind = sp[TG_SP_TURN], n = L.n;
    const int first = L.turn_first, ncp = L.turn_ncp, nint = ncp - 3, row = L.r_turn;
    const double al = x[L.ia];
    const double scale = kind == TG_TURN_CURVATURE ? 100.0 : 1.0;
    double *base = scr, *pa = scr + nint, *pert = scr + 2 * nint;
    const double ha = tg_fd_step(al, xl[L.ia], xu[L.ia]);
    // base and alpha-perturbed bound of every interval; then one item per (interval, coordinate, local control point)
    #pragma unroll 1
    for (int q = lane; q < 2 * nint + nint * 4 * D; q += TG_NL) {
        TgInterval<D> I;
        int j, pi = -1;
        double pv = 0, *dst;
        if (q < 2 * nint) {
            j = q < nint ? q : q - nint;
            dst = q < nint ? base + j : pa + j;
        } else {
            const int r = q - 2 * nint;
            j = r / (4 * D);
            const int cl = r - j * 4 * D, c = cl >> 2, l = cl & 3;
            pi = c * N + first + j + l;
            pv = x[pi] + tg_fd_step(x[pi], xl[pi], xu[pi]);
            dst = pert + (c * ncp + j + l) * 4 + l;
        }
        tg_load_interval<D>(x, N, first + j, I, pi, pv);
        *dst = tg_interval_turn_bound<D>(I, (q >= nint && q < 2 * nint) ? al + ha : al, kind, 0);
    }
    TG_SYNC();
    #pragma unroll 1
    for (int i = lane; i < n; i += TG_NL) {
        const int c = i / N, p = i - c * N - first;
        double entry = 0;
        if ((i < D * N && p >= 0 && p < ncp) || i == L.ia) {
            double best = 0;
            #pragma unroll 1
            for (int j = 0; j < nint; j++) {
                const int l = p - j;
                const double b = i == L.ia ? pa[j] : ((l >= 0 && l <= 3) ? pert[(c * ncp + p) * 4 + l] : base[j]);
                if (b > best) best = b;
            }
            const double cp = -((best - par[L.p_turn]) * scale);
            const double dx = (x[i] + tg_fd_step(x[i], xl[i], xu[i])) - x[i];
            entry = (cp - c0) / dx;
        }
        A[i * lda + row] = entry;
    }
    TG_SYNC();
}

// scr: K nint + 4 d N doubles (the first K nint are the base distances, as tg_rows_obstacles leaves them)
template <int D>
TG_EVAL_FN void tg_fd_obstacles(const TgLayout &L, const double *par, const double *x, const double *xl, const double *xu,
                           const double *cbase, double *A, int lda, int arow0, double *scr)
{
    // arow0: row of A that holds the first obstacle row (L.r_obs, or less when A stores no corridor rows)
    const int N = L.N, nint = L.nint, K = L.n_obs, lane = TG_LANE(), n = L.n;
    double *base = scr, *pert = scr + K * nint;
    #pragma unroll 1
    for (int q = lane; q < K * nint; q += TG_NL) {
        const int k = q / nint, j = q - k * nint;
        double ctr[D];
#pragma unroll
        for (int c = 0; c < D; c++) ctr[c] = par[L.p_obs_c + c * K + k];
        base[q] = tg_hull_distance<D>(x, N, j, ctr, par[L.p_obs_r + k], 0);
    }
    TG_SYNC();
    #pragma unroll 1
    for (int k = 0; k < K; k++) {
        double ctr[D];
#pragma unroll
        for (int c = 0; c < D; c++) ctr[c] = par[L.p_obs_c + c * K + k];
        const double rad = par[L.p_obs_r + k];
        #pragma unroll 1
        for (int r = lane; r < nint * 4 * D; r += TG_NL) {
            const int j = r / (4 * D), cl = r - j * 4 * D, c = cl >> 2, l = cl & 3;
            const int i = c * N + j + l;
            const double pv = x[i] + tg_fd_step(x[i], xl[i], xu[i]);
            pert[i * 4 + l] = tg_hull_distance<D>(x, N, j, ctr, rad, 0, i, pv);
        }
        TG_SYNC();
        #pragma unroll 1
        for (int i = lane; i < n; i += TG_NL) {
            double entry = 0;
            if (i < D * N) {
                const int p = i % N;
                double best = DBL_MAX;
                #pragma unroll 1
                for (int j = 0; j < nint; j++) {
                    const int l = p - j;
                    const double v = (l >= 0 && l <= 3) ? pert[i * 4 + l] : base[k * nint + j];
                    if (best > v) best = v;
                }
                const double dx = (x[i] + tg_fd_step(x[i], xl[i], xu[i])) - x[i];
                entry = (best - cbase[L.r_obs + k]) / dx;
            }
            A[i * lda + arow0 + k] = entry;
        }
        TG_SYNC();
    }
}

// constant Jacobian rows of the linear blocks (full-row sink only: compact == 0)
template <int D>
TG_FN void tg_linear_jacobian_d(const TgLayout &L, const int *sp, const double *par, const TgJac &J)
{
    tg_jac_location(L, sp, par, J);
    if (L.n_sfc && J.compact != 2) tg_jac_sfc<D>(L, sp, par, J);
    TG_SYNC();
}

#endif  // TG_EVAL_H
