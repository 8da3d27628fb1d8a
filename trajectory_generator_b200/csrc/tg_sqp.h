// Batched sequential quadratic programming: one warp runs the whole SLSQP
// iteration of one trajectory problem, replacing the per-problem
// scipy.optimize.minimize(method='SLSQP') call of the reference
// (TG/trajectory_generator.py:87-94; behaviour restated in SURVEY.md Appendix B,
// after D. Kraft, "A software package for sequential quadratic programming",
// DFVLR-FB 88-28, 1988).
//
// The outer iteration keeps SLSQP's semantics -- L1 merit function with the
// multiplier rule mu <- max(|lambda|, (mu+|lambda|)/2), Armijo-type line search
// with at most 10 quadratic-interpolation trials and alpha >= 0.1, Powell-damped
// BFGS applied as two rank-one updates of an LDL^T factorisation, reset of the
// factor when the merit's directional derivative is not negative (more than 5
// resets -> exit 8), both convergence tests, augmented subproblem (one slack,
// penalty 100, x10 up to 5 times) for inconsistent linearisations, bound
// clipping -- so that iterates follow the reference's on the same problem.
//
// The QP subproblem is strictly convex, so its solution and multipliers are
// unique; instead of SLSQP's LSQ/LSEI/LDP/NNLS chain it is solved with a dual
// active-set method (Goldfarb & Idnani 1983) that works directly on the
// maintained factor: J = L^-T D^-1/2, an orthogonal-triangular factor of the
// active normals (Householder on add, Givens on drop).  Jacobians are analytic
// (tg_eval.h), not finite differences.
//
// Every array lives in one per-problem workspace (shared memory on the device);
// lanes stride over vector entries / matrix rows.  Host build: one lane.
#ifndef TG_SQP_H
#define TG_SQP_H

#include "tg_eval.h"

struct TgSqpResult {
    int status, nit, nfev;
    double f;
};

// Per-problem state.  The PERSISTENT part survives between the two stages of an iteration (it lives in global
// memory when the stages run as separate lock-step kernels); the SCRATCH part is only used inside a stage.
struct TgSqpCtl {
    double f, f0, t0, h3, h4, alpha, acc;
    double flops;        // algorithmic fp64 operations of the QP stage so far (model counts, see tg_sqp_stage_qp)
    int state, iter, ireset, line, badlin, nfev, status, need_reset, maxiter, flags;
    int nract;           // rows (< m) with a non-zero multiplier after the last QP: W.ract[0 .. nract)
    int need_der;        // derivatives at the accepted point are still to be formed (stage DER)
    int pins_hold;       // the eliminated coordinates have reached their values (tg_sqp_stage_qp): their block of B is frozen
};
enum { TG_ST_INIT = 0, TG_ST_QP, TG_ST_LS, TG_ST_UPDATE, TG_ST_DONE };
#define TG_CTL_DOUBLES ((int)((sizeof(TgSqpCtl) + 7) / 8))

struct TgSqpWs {
    int n, n1, m, lda, ldq, nc;      // nc = m + 2*n1 (constraints incl. variable bounds); lda: rows of A (no corridor rows)
    int sfc0, nsfc, sfc_npts, cpN, cpd;      // corridor rows [sfc0, sfc0 + 2 nsfc): row -> interval -> the only non-zero columns
    // variables pinned by an equality row with a single entry (zero-velocity terminal waypoints pin three control
    // points per coordinate, CF/waypoint_constraints.py:122-147): eliminated from the QP subproblem, see tg_qp_solve.
    // ne of them (nf = n - ne stay); esk / eek: pins at the start / at the end; erow_s / erow_e: first pin row of each
    int ne, nf, esk, eek, rsk, rek, erow_s, erow_e;      // rsk / rek: rotated location triple at the start / at the end
    TgSqpCtl *ctl;
    // persistent
    double *x, *xl, *xu, *g, *s, *x0, *gl, *c, *mu, *r, *Lm, *Dd, *A;
    double *rot;         // persistent: rotation (d x d, row-major) of the corridor that owns each interval, written once by stage LS
    // scratch
    double *u, *v, *w, *cf, *Jq, *R, *rsub, *z, *dq, *rq, *np, *uq, *xq, *hw, *rdi, *scratch;
    double *rotq;        // scratch: copy of rot for the violation scans of the QP stage
    int *act;
    unsigned char *iact; // scratch: constraint (row or bound) is in the active set
    int *ract;           // persistent: active rows of the last QP, in the order they were added
    int *perm;           // scratch: QP order (free coordinates first, eliminated ones behind them) -> index in rotated space
    int *qix;            // scratch: the inverse (tg_qp_index of every index)
    double *sq;          // scratch (pinned variables only): the step in QP order, for the factor update
    double *usc;         // scratch of the factor update (5 n doubles) while the copy of L occupies J's storage
    int jsz;             // doubles of J's storage
    double *Ad;          // scratch (pinned variables only, else 0): copy of the dense inequality rows of A, row r at Ad + r n1
};

TG_HD int tg_odd(int v) { return v | 1; }

// number of variables the QP subproblem eliminates (pinned control points): 3 d per zero-velocity terminal waypoint
TG_HD int tg_sqp_pinned(const TgLayout &L)
{
#ifdef TG_NO_ELIM
    return 0;
#else
    if (L.d < 1 || L.N < 6) return 0;
    // 3 d per zero-velocity terminal waypoint (pins), d per plain location block (not the target form of the end
    // waypoint, whose rows carry the scale factor too: TG_SP_END_KIND == 2 has its velocity in the parameter row)
    // (other problem kinds that run the same stages -- the spline order converter -- have no such blocks: n_start = 0)
    int s = L.n_start == 3 * L.d ? 3 : L.n_start == L.d ? 1 : 0;
    int e = L.n_end == 3 * L.d ? 3 : (L.n_end == L.d && L.p_sdir == L.p_target_vel) ? 1 : 0;
    // A shape with pins keeps its plain location rows: the rotation costs every step of the subproblem a pass over the
    // step (rotated space <-> order of x), which the d rows less do not repay once the pins have shrunk the subproblem
    // (measured on C4: QP stage 133 ms with the pins alone, 147 ms with the start triples rotated as well).
    if (s == 3 || e == 3) { s = s == 3 ? 3 : 0; e = e == 3 ? 3 : 0; }
    return L.d * (s + e);
#endif
}
// variables of the (augmented) QP subproblem after the elimination: what the lanes of a group stride over
TG_HD int tg_sqp_qp_dim(const TgLayout &L) { return L.n - tg_sqp_pinned(L) + 1; }
TG_HD int tg_rp(int j) { return j * (j + 1) / 2; }      // offset of column j of the packed upper-triangular R

// unroll factor of the sequential inner products / updates of the QP stage (trip counts are n <= 62).  2 since the end
// of round 2 (was 4): the stage waits on instruction fetch, and the smaller loops are worth 0.6 % (C4) ... 1.2 % (C3);
// 1 loses 8 % on C3.
#ifndef TG_UNROLL_N
#define TG_UNROLL_N 2
#endif
// (Two interleaved accumulator chains per inner product -- even / odd terms, added at the end -- were measured in round 2:
// QP stage +-0 % on C3 / C4, +3 ... 5 % on C2 / C5: the chains are not what the stage waits on once the loads are counted.)
#define TG_PRAGMA_(x) _Pragma(#x)
#define TG_PRAGMA(x) TG_PRAGMA_(x)
#define TG_UNROLL_INNER TG_PRAGMA(unroll TG_UNROLL_N)
// lanes of the shuffle-based recurrences (a warp, or the 16 lanes of a group) and their mask
#define TG_SW (TG_GS >= 32 ? 32 : TG_GS)
#define TG_SMASK() (TG_GS >= 32 ? 0xffffffffu : TG_GMASK())
// loops over the m constraint values (c, mu: global memory when the kernel does not stage the state).  Unrolled by 4 --
// several loads in flight -- they cost C4's QP stage 2 %: its warps wait on instruction fetch before anything else.
// Unroll factors of a few more loops of the stage.  Its one-warp kernels wait on instruction fetch before anything else
// (profiles/README.md), and unrolling these loops costs more in fetches than it saves in issue slots -- measured on C4,
// 65,536 problems: products with the active rows behind the Lagrangian gradient 4 -> 1 and the scan of the copied dense
// rows 8 -> 1: QP stage 126 -> 110 ms; the recurrences 2 -> 1, the scan of dense rows in global memory 8 -> 2, the
// factor copies and the product for the pin multipliers 8 -> 2: 110 -> 107 ms.
// (the two-warp kernels do not wait on fetches -- C3 loses 2 % without the unrolling)
#ifndef TG_LAG_UNROLL
#define TG_LAG_UNROLL (TG_GS == 64 ? 4 : 1)
#endif
#ifndef TG_DENSE_UNROLL
#define TG_DENSE_UNROLL (TG_GS == 64 ? 8 : 1)
#endif
#ifndef TG_REC_UNROLL
#define TG_REC_UNROLL (TG_GS == 64 ? 2 : 1)
#endif
#ifndef TG_DENSE_FAR_UNROLL
#define TG_DENSE_FAR_UNROLL (TG_GS == 64 ? 8 : 2)
#endif
#ifndef TG_LAG_FAR_UNROLL
#define TG_LAG_FAR_UNROLL 2
#endif
#ifndef TG_VIOL_UNROLL
#define TG_VIOL_UNROLL 1
#endif

// The QP-stage functions are inlined into the lock-step QP kernel (one call site each; with the workspace carved
// from the kernel's shared array the compiler then knows the address space of every access).  The fused kernel's
// translation unit defines TG_SQP_NOINLINE (instruction-cache footprint).
#if defined(__CUDACC__) && !defined(TG_SQP_NOINLINE)
#define TG_QFN static __host__ __device__ __forceinline__
#else
#define TG_QFN TG_FN
#endif

// Carves the per-problem state.  The persistent block is [ctl | x xl xu g c | s x0 mu | gl r Dd | ract rot | A | Lm]; its first
// `npre` doubles (everything the line-search stage touches except A) may be staged at `prefix` while the rest
// stays at `pbase` (+ offset) -- pass prefix == pbase for one contiguous block.  The scratch block is
// [QP-stage scratch | evaluation scratch (cf, evaluators' scratch)]; `ebase` != 0 places the evaluation scratch
// elsewhere (the line-search kernel only allocates that part, the QP kernel only the first: *nsq_ doubles).
// Sizes come back in doubles.
TG_HD void tg_sqp_carve4(const TgLayout &L, double *prefix, double *pbase, double *sbase, double *ebase, TgSqpWs *W,
                         size_t *np_, size_t *ns_, size_t *npre_, size_t *nsq_)
{
    const int n = L.n, n1 = n + 1, m = L.m;
    TgSqpWs w;
    const int ma = m - 2 * L.n_sfc;       // rows stored in A
    w.n = n; w.n1 = n1; w.m = m; w.lda = tg_odd(ma > 0 ? ma : 1); w.ldq = tg_odd(n1); w.nc = m + 2 * n1;
    w.sfc0 = L.r_sfcl; w.nsfc = L.n_sfc; w.sfc_npts = 4 * L.nint; w.cpN = L.N; w.cpd = L.d;
    w.ne = tg_sqp_pinned(L); w.nf = n - w.ne;
    w.esk = w.ne && L.n_start == 3 * L.d; w.eek = w.ne && L.n_end == 3 * L.d; w.erow_s = L.r_start; w.erow_e = L.r_end;
    w.rsk = w.ne && !w.esk && !w.eek && L.n_start == L.d;
    w.rek = w.ne && !w.esk && !w.eek && L.n_end == L.d && L.p_sdir == L.p_target_vel;
    const int nqm = w.nf + 1;            // largest QP subproblem (augmented)
    if (w.ne) w.ldq = tg_odd(nqm);
    size_t o = 0;
    double *base = prefix;
#define TG_TAKE(field, count) w.field = base + o; o += (size_t)(count)
    w.ctl = (TgSqpCtl *)base; o += TG_CTL_DOUBLES;
    // (what the derivative stage touches first: its kernel stages [ctl .. c] only, tg_sqp_prefix_fd_doubles)
    TG_TAKE(x, n1); TG_TAKE(xl, n1); TG_TAKE(xu, n1); TG_TAKE(g, n1); TG_TAKE(c, m + 1);
    o += o & 1;
    TG_TAKE(s, n1); TG_TAKE(x0, n1); TG_TAKE(mu, m + 1);
    o += o & 1;                  // even counts: the staged pieces are moved with 16-byte accesses (double2 / 16-byte cp.async)
    if (npre_) *npre_ = o;
    base = pbase;
    TG_TAKE(gl, n1); TG_TAKE(r, w.nc + 1);
    TG_TAKE(Dd, n1);
    w.ract = (int *)(base + o); o += (size_t)(n1 / 2 + 1);
    TG_TAKE(rot, L.n_sfc ? L.nint * L.d * L.d : 0);
    TG_TAKE(A, w.lda * n1);
    o += o & 1;
    TG_TAKE(Lm, n * n);          // last: the lock-step QP kernel stages everything in front of it and leaves L in global memory
    o += o & 1;
    if (np_) *np_ = o;
    o = 0; base = sbase;
    TG_TAKE(u, n1); TG_TAKE(v, n1); TG_TAKE(w, n1);
    if (w.ne) { TG_TAKE(sq, n1); o += o & 1; } else w.sq = 0;
    // J (ldq x nqm) and R.  Pinned variables: the copy of L (n x n) that the factor update works on is larger than
    // the J of the smaller subproblem: it spans J, R and the five vectors behind them, and the update's 5 n doubles of
    // scratch come from the vectors behind those (uq .. rotq; the rotation table is copied again afterwards); J grows
    // by whatever the span lacks.
    const int rsz = w.ne ? nqm * (nqm + 1) / 2 + 1 : n1 * (n1 + 1) / 2 + 1;
    const int rotsz = L.n_sfc ? L.nint * L.d * L.d : 0;
    int jsz = w.ne ? w.ldq * nqm : w.ldq * n1;
    if (w.ne && jsz + rsz + 5 * n1 < n * n) jsz = n * n - rsz - 5 * n1;
    const int uscsz = w.ne ? (n1 + 1) + 3 * n1 + rotsz : 0;
    w.jsz = jsz;
    TG_TAKE(Jq, jsz);
    TG_TAKE(R, rsz);
    TG_TAKE(rsub, n1);      // R packed by columns (column j: rows 0..j at j(j+1)/2), its sub-diagonal during a drop
    TG_TAKE(z, n1); TG_TAKE(dq, n1); TG_TAKE(rq, n1); TG_TAKE(np, n1);
    w.usc = w.ne ? base + o : w.R;
    TG_TAKE(uq, n1 + 1); TG_TAKE(xq, n1); TG_TAKE(hw, n1);
    TG_TAKE(rdi, n1);
    TG_TAKE(rotq, rotsz);
    if (w.ne && uscsz < 5 * n) o += (size_t)(5 * n - uscsz);
    double *ints = base + o; o += (size_t)((n1 + 1 + (w.ne ? 2 * n1 : 0)) / 2 + 1);
    w.act = (int *)ints; w.perm = w.act + n1 + 1; w.qix = w.perm + n1;
    w.iact = (unsigned char *)(base + o); o += (size_t)((w.nc + 1 + 7) / 8);
    // (shapes with pinned variables run with their state in global memory -- C4 -- and scan the dense inequality rows
    // in every iteration of the QP: a copy next to the scratch)
    // (a few rows only: shapes with many dense rows are small ones, whose state the kernel stages anyway)
    const int nd = m - 2 * L.n_sfc - L.meq;
    if (w.ne && nd > 0 && nd <= 4) { TG_TAKE(Ad, nd * n1); } else w.Ad = 0;
    o += o & 1;
    if (nsq_) *nsq_ = o;
    if (ebase) { base = ebase - o; }
    // cf: constraint values at a perturbed point (finite-difference mode): the rows in front of the turning row only
    TG_TAKE(cf, L.r_turn + 1); TG_TAKE(scratch, tg_scratch_doubles(L));       // <- all the line-search stage needs
#undef TG_TAKE
    if (ns_) *ns_ = o;
    if (W) *W = w;
}

TG_HD void tg_sqp_carve3(const TgLayout &L, double *prefix, double *pbase, double *sbase, TgSqpWs *W, size_t *np_,
                         size_t *ns_, size_t *npre_)
{
    tg_sqp_carve4(L, prefix, pbase, sbase, 0, W, np_, ns_, npre_, 0);
}

TG_HD void tg_sqp_carve2(const TgLayout &L, double *pbase, double *sbase, TgSqpWs *W, size_t *np_, size_t *ns_)
{
    tg_sqp_carve3(L, pbase, pbase, sbase, W, np_, ns_, 0);
}

// scratch needed by the line-search stage alone (cf + the evaluators' scratch) / by the QP stage alone
TG_HD size_t tg_sqp_ls_scratch_doubles(const TgLayout &L) { return (size_t)L.r_turn + 1 + tg_scratch_doubles(L); }
// workspace slot of one lane group of the line-search / derivative kernels with their scratch in global memory: the
// evaluation scratch, padded to an even count (slots stay 16-byte aligned)
TG_HD size_t tg_sqp_ls_slot_doubles(const TgLayout &L) { const size_t e = tg_sqp_ls_scratch_doubles(L); return e + (e & 1); }
// front of the persistent block that the derivative stage touches: [ctl | x xl xu g | c], even
TG_HD size_t tg_sqp_prefix_fd_doubles(const TgLayout &L)
{
    const size_t o = (size_t)TG_CTL_DOUBLES + 4 * (size_t)(L.n + 1) + (size_t)L.m + 1;
    return o + (o & 1);
}
TG_HD size_t tg_sqp_qp_scratch_doubles(const TgLayout &L) { size_t a, b, c, d; tg_sqp_carve4(L, 0, 0, 0, 0, 0, &a, &b, &c, &d); return d; }
TG_HD size_t tg_sqp_prefix_doubles(const TgLayout &L) { size_t a, b, c; tg_sqp_carve3(L, 0, 0, 0, 0, &a, &b, &c); return c; }

// doubles the factor L occupies at the end of the persistent block (n^2 padded to an even count)
TG_HD size_t tg_sqp_factor_doubles(const TgLayout &L) { const size_t q = (size_t)L.n * L.n; return q + (q & 1); }

TG_HD size_t tg_sqp_persistent_doubles(const TgLayout &L) { size_t a, b; tg_sqp_carve2(L, 0, 0, 0, &a, &b); return a; }
TG_HD size_t tg_sqp_scratch_doubles(const TgLayout &L) { size_t a, b; tg_sqp_carve2(L, 0, 0, 0, &a, &b); return b; }
TG_HD size_t tg_sqp_workspace_doubles(const TgLayout &L) { return tg_sqp_persistent_doubles(L) + tg_sqp_scratch_doubles(L); }

// Shared memory of the lock-step stage kernels and the evaluation kernel (tg_kernels_solve.inc, tg_kernels_eval.inc):
// a CTA of TG_CTA_THREADS threads holds TG_CTA_THREADS / lanes lane groups.
#define TG_CTA_THREADS 128
// line-search / derivative stage, per lane group: [parameters | state prefix | evaluation scratch], every piece starting
// on a 16-byte boundary (the derivative stage stages the shorter prefix, tg_sqp_prefix_fd_doubles)
TG_HD size_t tg_ls_par_doubles(const TgLayout &L) { return ((size_t)L.P + 2) & ~(size_t)1; }
TG_HD size_t tg_ls_group_doubles(const TgLayout &L)
{
    const size_t n = tg_ls_par_doubles(L) + tg_sqp_prefix_doubles(L) + tg_sqp_ls_scratch_doubles(L);
    return n + (n & 1);
}
TG_HD size_t tg_fd_group_doubles(const TgLayout &L)
{
    const size_t n = tg_ls_par_doubles(L) + tg_sqp_prefix_fd_doubles(L) + tg_sqp_ls_scratch_doubles(L);
    return n + (n & 1);
}
TG_HD size_t tg_ls_smem_bytes(const TgLayout &L, int lanes) { return (size_t)(TG_CTA_THREADS / lanes) * tg_ls_group_doubles(L) * sizeof(double); }
TG_HD size_t tg_fd_smem_bytes(const TgLayout &L, int lanes) { return (size_t)(TG_CTA_THREADS / lanes) * tg_fd_group_doubles(L) * sizeof(double); }
// QP stage: the scratch, and with `staged` the persistent state except the factor L (which stays in global memory)
TG_HD size_t tg_qp_smem_bytes(const TgLayout &L, int lanes, int staged)
{
    const size_t state = staged ? tg_sqp_persistent_doubles(L) - tg_sqp_factor_doubles(L) : 0;
    return (size_t)(TG_CTA_THREADS / lanes) * (tg_sqp_qp_scratch_doubles(L) + state) * sizeof(double);
}
// evaluation kernel: lane groups of one CTA -- TG_CTA_THREADS / lanes, fewer where their shared memory exceeds the
// opt-in limit (long trajectories: 3-D with 8 x 63 corridor intervals needs 163 KB a group without `c`), 0 where not
// even one group fits
TG_HD int tg_eval_groups(const TgLayout &L, int lanes, bool sink_c, int smem_optin)
{
    const size_t fit = (size_t)smem_optin / (tg_eval_group_doubles(L, sink_c) * sizeof(double));
    return fit < (size_t)(TG_CTA_THREADS / lanes) ? (int)fit : TG_CTA_THREADS / lanes;
}

// one contiguous buffer: persistent part first, scratch behind it
TG_HD size_t tg_sqp_carve(const TgLayout &L, double *base, TgSqpWs *W)
{
    const size_t np_ = tg_sqp_persistent_doubles(L);
    size_t a, b;
    tg_sqp_carve2(L, base, base ? base + np_ : 0, W, &a, &b);
    return a + b;
}

TG_HD bool tg_finite(double v) { return v - v == 0; }

// ---------------------------------------------------------------------------
// A holds the Jacobian rows of every constraint EXCEPT the corridor rows (column i at A[i * lda + row], rows behind
// the corridor block moved up by 2 nsfc).  A corridor row (CF/sfc_constraints.py:53-77: lb <= R' Q <= ub on the
// MINVO points Q of an interval) has 4 d structural non-zeros, rot[rr][c] * M_minvo[l][k] at control point j + l of
// coordinate c; they are regenerated from the per-interval rotation table (written once by stage LS) -- the same
// product tg_jac_sfc forms -- instead of being stored: C4's state shrinks from 62 KB to 23 KB per problem.
// ---------------------------------------------------------------------------
TG_HD bool tg_is_sfc_row(const TgSqpWs &W, int p) { return p >= W.sfc0 && p < W.sfc0 + 2 * W.nsfc; }
TG_HD int tg_arow(const TgSqpWs &W, int p) { return p < W.sfc0 ? p : p - 2 * W.nsfc; }       // p not a corridor row

// entry (row p, column i < n) of a corridor row; rot: per-interval rotation table
TG_HD double tg_sfc_entry(const TgSqpWs &W, const double *rot, int p, int i)
{
    const int D = W.cpd, N = W.cpN, npts = W.sfc_npts;
    if (i >= D * N) return 0.0;
    int q = p - W.sfc0;
    const bool upper = q >= W.nsfc;
    if (upper) q -= W.nsfc;
    const int rr = q / npts, idx = q - rr * npts, j = idx >> 2, k = idx & 3;
    const int c = i / N, l = i - c * N - j;
    if (l < 0 || l > 3) return 0.0;
    const double v = rot[j * D * D + rr * D + c] * tg_minvo_py_t(l, k);
    return upper ? -v : v;
}

// ---------------------------------------------------------------------------
// Eliminated variables.  The terminal location rows are linear with constant coefficients, and the QP subproblem can
// be solved without them (null-space method):
//  * a zero-velocity terminal waypoint pins three control points per coordinate with rows that have a single entry 1
//    (tg_jac_location, kind 1): the step of such a variable is fixed, d_i = -c_i (zero once the pin holds);
//  * a plain location row reads [1/6 2/3 1/6] (P0, P1, P2) = b per coordinate (kind 0).  With H the 3 x 3 Householder
//    reflection that sends that row to -|w| e0, the rotated coordinates y = H (P0, P1, P2) have y0 pinned the same
//    way, d_y0 = -c / (-|w|), and y1, y2 free.
// The subproblem is then solved over the other nf coordinates only.  "Rotated space": x with every such triple replaced
// by H x_triple (H is symmetric and orthogonal: the same product maps back).  "QP order": the rotated coordinates, the
// eliminated ones LAST; the factor L D L' of B is kept in that order, so the factor of the free block is the
// leading block of L and D.  Same iterates in exact arithmetic.  C4: 34 -> 22 variables and 12 of its 15 equality
// rows gone, one warp per problem instead of two; C2 / C5: 17 -> 13, 4 of 8 equality rows gone.
// ---------------------------------------------------------------------------
#define TG_LOC_SIGMA (-0.70710678118654752440)       // the location row in rotated space: TG_LOC_SIGMA e0
TG_HD double tg_loc_h(int a, int b)
{
    // H = I - 2 v v' / v'v, v = w / |w| + e0, w = [1/6 2/3 1/6]
    const double h00 = -0.23570226039551584147, h01 = -0.94280904158206336587, h11 = 0.28066095096048549785,
                 h12 = -0.17983476225987862554, h22 = 0.95504130943503034362;
    const int lo = a < b ? a : b, hi = a < b ? b : a;
    return lo == 0 ? (hi == 1 ? h01 : h00) : lo == 1 ? (hi == 1 ? h11 : h12) : h22;
}
// eliminated coordinates per coordinate axis at the start / at the end
TG_HD int tg_elim_s(const TgSqpWs &W) { return 3 * W.esk + W.rsk; }
TG_HD int tg_elim_e(const TgSqpWs &W) { return 3 * W.eek + W.rek; }
TG_HD bool tg_is_pin_row(const TgSqpWs &W, int p)
{
    return ((W.esk | W.rsk) && p >= W.erow_s && p < W.erow_s + tg_elim_s(W) * W.cpd) ||
           ((W.eek | W.rek) && p >= W.erow_e && p < W.erow_e + tg_elim_e(W) * W.cpd);
}
// first variable of the rotated triple that holds variable i of x, -1 if it is not in one
TG_HD int tg_rot_base(const TgSqpWs &W, int i)
{
    const int N = W.cpN;
    if (!(W.rsk | W.rek) || i >= W.cpd * N) return -1;
    const int c = i / N, j = i - c * N;
    if (W.rsk && j < 3) return c * N;
    if (W.rek && j >= N - 3) return c * N + N - 3;
    return -1;
}
// entry i of a vector of x taken to rotated space
TG_HD double tg_rot_get(const TgSqpWs &W, const double *vec, int i)
{
    const int b = tg_rot_base(W, i);
    if (b < 0) return vec[i];
    const int a = i - b;
    return tg_loc_h(a, 0) * vec[b] + tg_loc_h(a, 1) * vec[b + 1] + tg_loc_h(a, 2) * vec[b + 2];
}
// coordinate i of rotated space (same index as the variable of x it replaces) -> position in QP order (free
// coordinates keep their order; eliminated ones follow, ascending)
TG_HD int tg_qp_index(const TgSqpWs &W, int i)
{
    if (!W.ne) return i;
    const int N = W.cpN, es = tg_elim_s(W), ee = tg_elim_e(W), per = es + ee;
    if (i >= W.cpd * N) return i - W.cpd * per;
    const int c = i / N, j = i - c * N;
    if (j < es) return W.nf + c * per + j;                                   // pins j = 0..2, or y0 of the rotated triple
    if (ee && j >= N - 3 && j < N - 3 + ee) return W.nf + c * per + es + (j - (N - 3));
    return i - c * per - es - (j >= N - 3 ? ee : 0);
}
// eliminated coordinate e (QP position nf + e) -> its row, and the row's entry there
TG_HD int tg_pin_row(const TgSqpWs &W, int e)
{
    const int es = tg_elim_s(W), per = es + tg_elim_e(W), c = e / per, t = e - c * per;
    return t < es ? W.erow_s + es * c + t : W.erow_e + tg_elim_e(W) * c + (t - es);
}
TG_HD double tg_pin_sigma(const TgSqpWs &W, int e)
{
    const int es = tg_elim_s(W), per = es + tg_elim_e(W), t = e % per;
    return (t < es ? W.rsk : W.rek) ? TG_LOC_SIGMA : 1.0;
}

// coefficient of the slack variable of the augmented problem in row j (SLSQP: -c for equalities, max(-c, 0) else)
TG_HD double tg_slack_coeff(const TgSqpWs &W, int meq, int j) { return j < meq ? -W.c[j] : fmax(-W.c[j], 0.0); }

// ---------------------------------------------------------------------------
// LDL^T rank-one update  B <- B + sigma z z^T  (composite-t method of Fletcher &
// Powell, as used by SLSQP's LDL routine).  Lm: unit lower factor, column i at
// Lm[i*n + j] (j > i); Dd: diagonal.  z is destroyed; w is scratch (n), sc is
// scratch (5 n).
//
// SLSQP's loop over the columns carries three divisions per column (delta = v/d,
// alpha = t'/t, beta = delta/t') behind the recurrence v <- v - v_i L_i.  The
// same numbers are formed here in three phases so that no division sits on a
// serial path: (A) the recurrence alone -- v = L^-1 z, one step per column;
// (B) the scalars of every column at once, one column per lane (the only serial
// part left is the chain t' = t + delta v of multiply-adds; for sigma < 0 the
// forward / backward sums of v^2/d); (C) the columns of L, one per lane, each
// lane re-running its own entry of the recurrence (same operations, same
// order: bit-identical to the one-loop form).
// ---------------------------------------------------------------------------
#ifdef __CUDA_ARCH__
#define TG_MULADD2(a, b, c, d) fma((a), (b), __dmul_rn((c), (d)))      // a b + c d, contracted the way the one-loop form was
#else
#define TG_MULADD2(a, b, c, d) ((a) * (b) + (c) * (d))
#endif
// (ld: stride of the columns of Lm -- the update of the leading n x n block of a larger factor)
TG_QFN void tg_ldl_update(int n, double sigma, double *z, double *Lm, double *Dd, double *w, double *sc, int ld)
{
    const int lane = TG_LANE();
    if (sigma == 0) return;
    double *vf = w, *dl = sc, *tpv = sc + n, *al = sc + 2 * n, *be = sc + 3 * n, *ga = sc + 4 * n;
    double t = 1 / sigma;
    // ---- A: vf = L^-1 z
    #pragma unroll 1
    for (int i = lane; i < n; i += TG_NL) vf[i] = z[i];
    TG_SYNC();
#if defined(__CUDA_ARCH__) && TG_GS >= 16
    // one warp (or half of one: 16-lane groups), v in registers (entries lane and lane + TG_SW), the pivot handed round
    // with a shuffle (see the back substitution of tg_qp_directions); same operations in the same order.
    // n > 2 TG_SW: the shared-memory form.
    if (n > 2 * TG_SW) {
        if (TG_SERIAL_ACTIVE()) {
            #pragma unroll 1
            for (int i = 0; i < n - 1; i++) {
                const double vv = vf[i];
                #pragma unroll 1
                for (int j = i + 1 + lane; j < n; j += TG_SERIAL_LANES) vf[j] -= vv * Lm[i * ld + j];
                TG_SERIAL_SYNC();
            }
        }
    } else if (TG_SERIAL_ACTIVE()) {
        const int l32 = lane & (TG_SW - 1);
        double v0 = l32 < n ? vf[l32] : 0.0, v1 = l32 + TG_SW < n ? vf[l32 + TG_SW] : 0.0;
        TG_PRAGMA(unroll TG_REC_UNROLL)
        for (int i = 0; i < n - 1; i++) {
            const double vv = __shfl_sync(TG_SMASK(), i < TG_SW ? v0 : v1, i & (TG_SW - 1), TG_SW);
            const double *Li = Lm + i * ld;
            if (l32 > i && l32 < n) v0 -= vv * Li[l32];
            if (l32 + TG_SW > i && l32 + TG_SW < n) v1 -= vv * Li[l32 + TG_SW];
        }
        if (l32 < n) vf[l32] = v0;
        if (l32 + TG_SW < n) vf[l32 + TG_SW] = v1;
    }
#else
    if (TG_SERIAL_ACTIVE()) {
        #pragma unroll 1
        for (int i = 0; i < n - 1; i++) {
            const double vv = vf[i];
            #pragma unroll 1
            for (int j = i + 1 + lane; j < n; j += TG_SERIAL_LANES) vf[j] -= vv * Lm[i * ld + j];
            TG_SERIAL_SYNC();
        }
    }
#endif
    TG_SYNC();
    // ---- B: delta_i = v_i / d_i ; t'_i ; alpha_i = t'_i / t_i, beta_i = delta_i / t'_i, gamma_i = t_i / t'_i
    #pragma unroll 1
    for (int i = lane; i < n; i += TG_NL) {
        const double vv = vf[i], di = Dd[i];
        dl[i] = vv / di;
        if (sigma < 0) al[i] = vv * vv / di;
    }
    TG_SYNC();
    const double tstart = sigma < 0 ? 0 : t;
    if (sigma < 0) {
        #pragma unroll 1
        for (int i = 0; i < n; i++) t += al[i];
        if (t >= 0) t = DBL_EPSILON / sigma;
        #pragma unroll 1
        for (int i = n - 1; i >= 0; i--) {
            if (lane == 0) tpv[i] = t;
            t -= al[i];
        }
    } else {
        #pragma unroll 1
        for (int i = 0; i < n; i++) {
            t = t + dl[i] * vf[i];
            if (lane == 0) tpv[i] = t;
        }
    }
    const double t0 = sigma < 0 ? t : tstart;            // t before column 0
    TG_SYNC();
    #pragma unroll 1
    for (int i = lane; i < n; i += TG_NL) {
        const double tp = tpv[i], ti = i ? tpv[i - 1] : t0;
        const double alpha = tp / ti;
        be[i] = dl[i] / tp;
        ga[i] = ti / tp;
        al[i] = alpha;
        Dd[i] = alpha * Dd[i];
    }
    TG_SYNC();
    // ---- C: column j of L and its own entry of the recurrence
    #pragma unroll 1
    for (int j = 1 + lane; j < n; j += TG_NL) {
        double zj = z[j];
        TG_PRAGMA(unroll TG_REC_UNROLL)
        for (int i = 0; i < j; i++) {
            const double uu = Lm[i * ld + j], vv = vf[i], beta = be[i];
            if (al[i] > 4) {
                Lm[i * ld + j] = TG_MULADD2(ga[i], uu, beta, zj);
                zj -= vv * uu;
            } else {
                zj -= vv * uu;
                Lm[i * ld + j] = uu + beta * zj;
            }
        }
    }
    TG_SYNC();
}

// out = L D L^T s  (tmp: n scratch)
TG_QFN void tg_ldl_apply(int n, const double *Lm, const double *Dd, const double *s, double *tmp, double *out, int ld)
{
    const int lane = TG_LANE();
    #pragma unroll 1
    for (int i = lane; i < n; i += TG_NL) {
        double h = s[i];
        TG_UNROLL_INNER
        for (int j = i + 1; j < n; j++) h += Lm[i * ld + j] * s[j];
        tmp[i] = Dd[i] * h;
    }
    TG_SYNC();
    #pragma unroll 1
    for (int i = lane; i < n; i += TG_NL) {
        double h = tmp[i];
        TG_UNROLL_INNER
        for (int j = 0; j < i; j++) h += Lm[j * ld + i] * tmp[j];
        out[i] = h;
    }
    TG_SYNC();
}

// entries i0 .. n-1 of L D L^T s with L in global memory (the multipliers of the eliminated coordinates at the end of
// a subproblem): more loads in flight, and only the rows that are asked for in the second product
TG_QFN void tg_ldl_apply_tail(int n, const double *Lm, const double *Dd, const double *s, double *tmp, double *out, int ld, int i0)
{
    const int lane = TG_LANE();
    #pragma unroll 1
    for (int i = lane; i < n; i += TG_NL) {
        double h = s[i];
        #pragma unroll 2
        for (int j = i + 1; j < n; j++) h += Lm[i * ld + j] * s[j];
        tmp[i] = Dd[i] * h;
    }
    TG_SYNC();
    #pragma unroll 1
    for (int i = i0 + lane; i < n; i += TG_NL) {
        double h = tmp[i];
        #pragma unroll 2
        for (int j = 0; j < i; j++) h += Lm[j * ld + i] * tmp[j];
        out[i] = h;
    }
    TG_SYNC();
}

// ---------------------------------------------------------------------------
// QP subproblem:  min 1/2 s'Bs + g's   s.t.  A_eq s + c_eq = 0,  A_in s + c_in >= 0,  u <= s <= v
// with B = L D L' (dimension n) plus, for the augmented problem (nq = n+1), a
// last diagonal entry rho.  Non-finite u/v entries mean "no bound".
// Output: W.xq (step), W.r (multipliers of rows, lower bounds, upper bounds).
// returns 1 solved (SLSQP's LSQ mode 1), 4 inconsistent constraints, 6 dependent
// equality normals, 3 iteration limit.
// ---------------------------------------------------------------------------
#define TG_QP_OK 1

// entry i (a variable of x; i == n: the slack of the augmented problem) of the normal of row / bound p
TG_HD double tg_normal_entry(const TgSqpWs &W, int meq, int p, int i)
{
    if (p < W.m) {
        if (tg_is_sfc_row(W, p)) return i < W.n ? tg_sfc_entry(W, W.rotq, p, i) : tg_slack_coeff(W, meq, p);
        return W.A[i * W.lda + tg_arow(W, p)];
    }
    const int q = p - W.m;
    const int i0 = q < W.n1 ? q : q - W.n1;
    return i == i0 ? (q < W.n1 ? 1.0 : -1.0) : 0.0;
}

// the same in rotated space (tg_rot_get of the normal)
TG_HD double tg_normal_entry_r(const TgSqpWs &W, int meq, int p, int i)
{
    const int b = i < W.n ? tg_rot_base(W, i) : -1;
    if (b < 0) return tg_normal_entry(W, meq, p, i);
    const int a = i - b;
    return tg_loc_h(a, 0) * tg_normal_entry(W, meq, p, b) + tg_loc_h(a, 1) * tg_normal_entry(W, meq, p, b + 1) +
           tg_loc_h(a, 2) * tg_normal_entry(W, meq, p, b + 2);
}

// ELIM: entry k of the QP's vectors is coordinate perm[k] of rotated space (k < nf) or the slack (k == nf)
#define TG_XI(k) (ELIM ? ((k) < W.nf ? W.perm[k] : W.n) : (k))

template <bool ELIM>
TG_HD void tg_qp_normal(const TgSqpWs &W, int nq, int meq, int p, double *np, bool coupled)
{
    const int lane = TG_LANE();
    if (ELIM) {
        // the normal in the order of x first (W.hw: free until tg_qp_directions), one entry per lane; then rotated space
        #pragma unroll 1
        for (int i = lane; i <= W.n; i += TG_NL) W.hw[i] = (i < W.n || nq > W.nf) ? tg_normal_entry(W, meq, p, i) : 0.0;
        TG_SYNC();
        #pragma unroll 1
        for (int k = lane; k < nq; k += TG_NL) {
            double h = k < W.nf ? tg_rot_get(W, W.hw, W.perm[k]) : W.hw[W.n];
            if (coupled && k == W.nf)        // the slack moves the eliminated coordinates along c_P / sigma (W.w)
                #pragma unroll 1
                for (int e = 0; e < W.ne; e++) h += tg_rot_get(W, W.hw, W.perm[W.nf + e]) * W.w[e];
            np[k] = h;
        }
    } else if (p < W.m && tg_is_sfc_row(W, p)) {
        #pragma unroll 1
        for (int i = lane; i < nq; i += TG_NL) np[i] = i < W.n ? tg_sfc_entry(W, W.rotq, p, i) : tg_slack_coeff(W, meq, p);
    } else if (p < W.m) {
        const int pa = tg_arow(W, p);
        #pragma unroll 1
        for (int i = lane; i < nq; i += TG_NL) np[i] = W.A[i * W.lda + pa];
    } else {
        const int q = p - W.m;
        const int i0 = q < W.n1 ? q : q - W.n1;
        const double sg = q < W.n1 ? 1.0 : -1.0;
        #pragma unroll 1
        for (int i = lane; i < nq; i += TG_NL) np[i] = i == i0 ? sg : 0.0;
    }
    TG_SYNC();
}

// value of constraint p at the current point of the QP (lane-parallel reduction; same result on all lanes).  W.np holds
// the normal of p (tg_qp_normal): row p of A is not read a second time.  ELIM: the point in QP coordinates is W.sq
// (W.xq is its image in the order of x, for the scans); `pins`: some eliminated coordinate has a non-zero step -W.w
// (the slack's share of it, in the augmented problem, is part of np[nf])
template <bool ELIM>
TG_HD double tg_qp_value(const TgSqpWs &W, int nq, int meq, int p, bool pins)
{
    if (p < W.m) {
        double s = 0;
        #pragma unroll 1
        for (int i = TG_LANE(); i < nq; i += TG_NL) s += W.np[i] * (ELIM ? W.sq[i] : W.xq[i]);
        if (ELIM && pins) {
            #pragma unroll 1
            for (int e = TG_LANE(); e < W.ne; e += TG_NL) s -= tg_normal_entry_r(W, meq, p, W.perm[W.nf + e]) * W.w[e];
        }
        return tg_wsum(s) + W.c[p];
    }
    const int q = p - W.m;
    return q < W.n1 ? W.xq[q] - W.u[q] : W.v[q - W.n1] - W.xq[q - W.n1];
}

// ELIM: a vector of QP coordinates y (free ones; the eliminated coordinate e has the value es W.w[e]) taken to the order
// of x: entry i of the result.  rb: tg_rot_base(W, i).
TG_HD double tg_qp_x_entry(const TgSqpWs &W, const double *y, double es, int i, int rb)
{
    if (rb < 0) { const int k = W.qix[i]; return k < W.nf ? y[k] : es * W.w[k - W.nf]; }
    const int a = i - rb;
    double h = 0;
    #pragma unroll
    for (int l = 0; l < 3; l++) { const int k = W.qix[rb + l]; h += tg_loc_h(a, l) * (k < W.nf ? y[k] : es * W.w[k - W.nf]); }
    return h;
}

// d = J' np ; z = J2 d2 ; rq = R^-1 d1 ; returns |d2|^2 (= z.np) and |d|^2
TG_QFN void tg_qp_directions(const TgSqpWs &W, int nq, int iq, double &d2n, double &dn)
{
    // (visiting only the non-zero entries of a sparse normal -- a bit mask of them, one bit scan per term -- was
    // measured: same numbers, QP stage +2 .. 3 % on C2 / C4: the stage is bound by dependent latency, not by issue slots)
    const int lane = TG_LANE(), ld = W.ldq;
    double a = 0, b = 0;
    #pragma unroll 1
    for (int k = lane; k < nq; k += TG_NL) {
        double h = 0;
        const double *col = W.Jq + k * ld;
        TG_UNROLL_INNER
        for (int i = 0; i < nq; i++) h += col[i] * W.np[i];
        W.dq[k] = h;
        W.hw[k] = h;
        if (k >= iq) a += h * h;
        b += h * h;
    }
    tg_wsum2(a, b);
    d2n = a; dn = b;
    TG_SYNC();
    // (64-lane groups: forming z on the second warp while the first runs the back substitution below was measured
    // neutral, +-0.5 %)
    #pragma unroll 1
    for (int i = lane; i < nq; i += TG_NL) {
        double h = 0;
        TG_UNROLL_INNER
        for (int k = iq; k < nq; k++) h += W.Jq[k * ld + i] * W.dq[k];
        W.z[i] = h;
    }
    // back substitution R rq = d1 (column oriented; hw holds the running right-hand side, rdi = 1 / diag R)
#if defined(__CUDA_ARCH__) && TG_GS >= 16
    // One warp (half of one: 16-lane groups), the running right-hand side in registers (entries lane and lane + TG_SW),
    // the pivot handed round with a shuffle: no shared-memory round trip and no warp sync per step.  Same operations in
    // the same order.  (More than 2 TG_SW active constraints: the shared-memory form below.)
    if (iq > 2 * TG_SW) {
        if (TG_SERIAL_ACTIVE()) {
            #pragma unroll 1
            for (int j = iq - 1; j >= 0; j--) {
                const double rj = W.hw[j] * W.rdi[j];
                if (lane == 0) W.rq[j] = rj;
                #pragma unroll 1
                for (int k = lane; k < j; k += TG_SERIAL_LANES) W.hw[k] -= W.R[tg_rp(j) + k] * rj;
                TG_SERIAL_SYNC();
            }
        }
    } else if (TG_SERIAL_ACTIVE()) {
        const int l32 = lane & (TG_SW - 1);
        double h0 = l32 < iq ? W.hw[l32] : 0.0, h1 = l32 + TG_SW < iq ? W.hw[l32 + TG_SW] : 0.0;
        TG_PRAGMA(unroll TG_REC_UNROLL)
        for (int j = iq - 1; j >= 0; j--) {
            const double rj = __shfl_sync(TG_SMASK(), j < TG_SW ? h0 : h1, j & (TG_SW - 1), TG_SW) * W.rdi[j];
            const double *Rj = W.R + tg_rp(j);
            if (l32 == (j & (TG_SW - 1))) W.rq[j] = rj;
            if (l32 < j) h0 -= Rj[l32] * rj;
            if (l32 + TG_SW < j) h1 -= Rj[l32 + TG_SW] * rj;
        }
    }
#else
    if (TG_SERIAL_ACTIVE()) {
        #pragma unroll 1
        for (int j = iq - 1; j >= 0; j--) {
            const double rj = W.hw[j] * W.rdi[j];
            if (lane == 0) W.rq[j] = rj;
            #pragma unroll 1
            for (int k = lane; k < j; k += TG_SERIAL_LANES) W.hw[k] -= W.R[tg_rp(j) + k] * rj;
            TG_SERIAL_SYNC();
        }
    }
#endif
    TG_SYNC();
}

// append the constraint with J'np = dq to the factorisation: Householder reflection of dq[iq..] onto e_iq applied
// to the columns iq.. of J.  J2 w = z - sigma J[:, iq] with z = J2 d2 from tg_qp_directions (d2n = |d2|^2).
TG_QFN void tg_qp_add(const TgSqpWs &W, int nq, int iq, double d2n)
{
    const int lane = TG_LANE(), ld = W.ldq;
    const double d0 = W.dq[iq];
    const double sigma = d0 > 0 ? -sqrt(d2n) : sqrt(d2n);
    // w = d2 - sigma e1 ;  w'w = 2 (|d2|^2 - sigma d0)
    const double ww = 2 * (d2n - sigma * d0);
    const double w0 = d0 - sigma;
    TG_SYNC();
    if (ww > 0) {
        const double sc = 2 / ww;
        #pragma unroll 1
        for (int i = lane; i < nq; i += TG_NL) {
            const double t = (W.z[i] - sigma * W.Jq[iq * ld + i]) * sc;
            W.Jq[iq * ld + i] -= t * w0;
            TG_UNROLL_INNER
            for (int k = iq + 1; k < nq; k++) W.Jq[k * ld + i] -= t * W.dq[k];
        }
    }
    #pragma unroll 1
    for (int k = lane; k < iq; k += TG_NL) W.R[tg_rp(iq) + k] = W.dq[k];
    if (lane == 0) {
        const double rd = ww > 0 ? sigma : d0;
        W.R[tg_rp(iq) + iq] = rd;
        W.rdi[iq] = 1 / rd;
    }
    TG_SYNC();
}

// remove the constraint at position l of the active list
TG_QFN void tg_qp_drop(const TgSqpWs &W, int nq, int &iq, int l)
{
    const int lane = TG_LANE(), ld = W.ldq;
    if (lane == 0) W.iact[W.act[l]] = 0;
    #pragma unroll 1
    for (int k = l; k < iq - 1; k++) {
        #pragma unroll 1
        for (int i = lane; i <= k + 1; i += TG_NL) {
            const double e = W.R[tg_rp(k + 1) + i];
            if (i <= k) W.R[tg_rp(k) + i] = e; else W.rsub[k] = e;          // row k+1 of the shifted column: to be rotated away
        }
        if (lane == 0) { W.act[k] = W.act[k + 1]; W.uq[k] = W.uq[k + 1]; }
        TG_SYNC();
    }
    iq--;
    #pragma unroll 1
    for (int j = l; j < iq; j++) {
        double cc = W.R[tg_rp(j) + j], ss = W.rsub[j];
        const double h = sqrt(cc * cc + ss * ss);
        TG_SYNC();
        if (h == 0) { if (lane == 0) W.rdi[j] = INFINITY; continue; }
        cc /= h; ss /= h;
        if (lane == 0) { W.R[tg_rp(j) + j] = h; W.rsub[j] = 0; W.rdi[j] = 1 / h; }
        #pragma unroll 1
        for (int k = j + 1 + lane; k < iq; k += TG_NL) {
            const double t1 = W.R[tg_rp(k) + j], t2 = W.R[tg_rp(k) + j + 1];
            W.R[tg_rp(k) + j] = cc * t1 + ss * t2;
            W.R[tg_rp(k) + j + 1] = -ss * t1 + cc * t2;
        }
        #pragma unroll 1
        for (int i = lane; i < nq; i += TG_NL) {
            const double t1 = W.Jq[j * ld + i], t2 = W.Jq[(j + 1) * ld + i];
            W.Jq[j * ld + i] = cc * t1 + ss * t2;
            W.Jq[(j + 1) * ld + i] = -ss * t1 + cc * t2;
        }
        TG_SYNC();
    }
    TG_SYNC();
}

// ELIM (pinned variables, see tg_is_pin_row): nq = nf (+ 1) variables in QP order; W.xq, W.g, W.u, W.v, A keep the
// order of x.  Lsrc / W.Lm / W.Dd: the factor of B in QP order.
template <bool ELIM>
TG_QFN int tg_qp_solve(const TgSqpWs &W, const double *Lsrc, int nq, int meq, double rho, double &fl, int &nract, double dfloor,
                       bool ident, bool hold, bool &moving)
{
    const int lane = TG_LANE(), ld = W.ldq, m = W.m;
    const int n = ELIM ? W.nf : W.n;            // variables of the plain subproblem
    const int nx = nq > n ? W.n1 : W.n;         // entries of xq (order of x; the slack is entry W.n)
    const int nc = m + 2 * W.n1;
    bool pins = false;                          // ELIM: some pinned variable still has to move
    double dslack = rho * rho;                  // ELIM, augmented problem while pins move: the slack's entry of D
    if (ELIM) {
        // A pin that is off by rounding alone (|c| <= 16 ulp of the variable: what x + (b - x) leaves behind) is put
        // right by the step like any other, but its products with B and its multiplier -- 1e-16 relative to the
        // gradient and to the merit function -- are not formed.
        #pragma unroll 1
        for (int e = lane; e < W.ne; e += TG_NL) {
            const double sg = tg_pin_sigma(W, e);
            const double cv = W.c[tg_pin_row(W, e)] / sg;       // residual of the coordinate itself
            const int i = W.perm[W.nf + e];
            const double xs = sg == 1.0 ? fabs(W.x[i]) : fabs(W.x[i]) + fabs(W.x[i + 1]) + fabs(W.x[i + 2]);
            W.w[e] = cv;
            if (fabs(cv) > 16 * 2.220446049250313e-16 * xs) pins = true;
        }
        pins = tg_any(pins) && !hold;       // (hold: they have reached their values before; their block of B is frozen)
    }
    moving = pins;
    const bool coupled = ELIM && pins && nq > n;      // the slack's column of J is not a unit vector
    if (ELIM && pins) {
        // W.sq = B [0; d_P], d_P = -c_P: what the pinned variables' fixed step adds to the gradient of the free ones
        // (only until the pins hold -- the first iterations).  `ident`: the factor has just been reset, B = I.
        // (before the packed copy is made: Lsrc may be the copy of L next to J, and the vectors used are outside it)
        #pragma unroll 1
        for (int k = lane; k < W.n; k += TG_NL) { W.hw[k] = k < W.nf ? 0.0 : -W.w[k - W.nf]; if (ident) W.sq[k] = W.hw[k]; }
        TG_SYNC();
        if (!ident) tg_ldl_apply(W.n, Lsrc, W.Dd, W.hw, W.rdi, W.sq, W.n);
    }
    const double EPS_DEP = 1e-26;     // |d2|^2 <= EPS_DEP |d|^2 : normal lies in the span of the active ones
    // ---- J = L^-T D^-1/2 (upper triangular), augmented entry 1/rho.  L is read n^2/2 times per lane: copy it next
    //      to J first (the storage of R is free until the first constraint is added)
    // (packed: row i of the copy holds L[i][j], j > i, at i npk - i (i + 1) / 2 - i - 1 + j)
    double *Ls = W.R;
    const int npk = coupled ? nq : n;                 // rows of the packed copy (coupled: + the slack's row, below)
    if (ELIM && Lsrc == W.Jq) {
        // The copy of L that the factor update left behind spans J's storage, R's and the vectors behind them (tg_sqp_carve4):
        // its entries that lie in R's storage are set aside first (W.usc: outside the span), then the packed copy is
        // written.  From here on the span is free; whatever else needs L reads W.Lm.
        double *tmp = W.usc;
        int toff = 0;
        #pragma unroll 1
        for (int i = 0; i < n - 1; i++) {
            int j0 = W.jsz - i * W.n;
            if (j0 < i + 1) j0 = i + 1;
            #pragma unroll 1
            for (int j = j0 + lane; j < n; j += TG_NL) tmp[toff + j - j0] = Lsrc[i * W.n + j];
            if (j0 < n) toff += n - j0;
        }
        TG_SYNC();
        toff = 0;
        #pragma unroll 1
        for (int i = 0; i < n - 1; i++) {
            const int bi = i * npk - i * (i + 1) / 2 - i - 1;
            int j0 = W.jsz - i * W.n;
            if (j0 < i + 1) j0 = i + 1;
            #pragma unroll 1
            for (int j = i + 1 + lane; j < n; j += TG_NL) Ls[bi + j] = j < j0 ? Lsrc[i * W.n + j] : tmp[toff + j - j0];
            if (j0 < n) toff += n - j0;
        }
    } else {
        #pragma unroll 1
        for (int i = 0; i < n - 1; i++) {
            const int bi = i * npk - i * (i + 1) / 2 - i - 1;
            #pragma unroll 1
            for (int j = i + 1 + lane; j < n; j += TG_NL) Ls[bi + j] = Lsrc[i * W.n + j];
        }
    }
    TG_SYNC();
    if (ELIM) {
        #pragma unroll 1
        for (int k = lane; k < nq; k += TG_NL) W.rq[k] = k < W.nf ? tg_rot_get(W, W.g, W.perm[k]) : W.g[W.n];       // gradient in QP order
        TG_SYNC();
        if (pins) {
            // g_f + B_fP d_P = g_f + (B [0; d_P])_f
            #pragma unroll 1
            for (int k = lane; k < W.nf; k += TG_NL) W.rq[k] += W.sq[k];
            TG_SYNC();
            if (coupled) {
                // Augmented problem: the pin rows read d_P = -(1 - slack) c_P, so the slack moves the pinned variables
                // along c_P.  In the variables [d_f; slack] the Hessian gains the row [B_fP c_P, c_P' B_PP c_P + rho^2]:
                // its factor is the free block's plus one row l = L_Pf' c_P with D entry rho^2 + |D_P^1/2 L_PP' c_P|^2,
                // and the slack's gradient entry is c_P' (g + B [0; d_P])_P.
                double gsl = 0, dd = 0;
                #pragma unroll 1
                for (int e = lane; e < W.ne; e += TG_NL) {
                    gsl += W.w[e] * (tg_rot_get(W, W.g, W.perm[W.nf + e]) + W.sq[W.nf + e]);
                    double h = W.w[e];
                    if (!ident)
                        #pragma unroll 1
                        for (int e2 = e + 1; e2 < W.ne; e2++) h += W.Lm[(W.nf + e) * W.n + W.nf + e2] * W.w[e2];
                    dd += W.Dd[W.nf + e] * h * h;
                }
                tg_wsum2(gsl, dd);
                dslack += dd;
                #pragma unroll 1
                for (int k = lane; k < W.nf; k += TG_NL) {
                    double h = 0;
                    if (!ident)
                        #pragma unroll 1
                        for (int e = 0; e < W.ne; e++) h += W.Lm[k * W.n + W.nf + e] * W.w[e];
                    Ls[k * npk - k * (k + 1) / 2 - k - 1 + W.nf] = h;
                }
                if (lane == 0) W.rq[W.nf] += gsl;
                TG_SYNC();
            }
        }
    }
    #pragma unroll 1
    for (int k = lane; k < nq; k += TG_NL) {
        double *col = W.Jq + k * ld;
        for (int i = 0; i < nq; i++) col[i] = 0;
        if (k < n || coupled) {
            col[k] = 1;
            #pragma unroll 1
            for (int i = k - 1; i >= 0; i--) {
                double h = 0;
                const double *Li = Ls + (i * npk - i * (i + 1) / 2 - i - 1);
                TG_UNROLL_INNER
                for (int j = i + 1; j <= k; j++) h += Li[j] * col[j];
                col[i] = -h;
            }
            const double sc = 1 / sqrt(fmax(k < n ? W.Dd[k] : dslack, dfloor));
            for (int i = 0; i <= k; i++) col[i] *= sc;
        } else col[k] = 1 / rho;      // SLSQP's LSQ puts rho itself (not its root) on the diagonal of E: penalty rho^2/2 delta^2
    }
    #pragma unroll 1
    for (int p = lane; p < nc; p += TG_NL) { W.iact[p] = 0; W.r[p] = 0; }
    const int nd = W.m - 2 * W.nsfc - meq;      // dense inequality rows
    if (ELIM && nd > 0 && nd <= 4) {
        #pragma unroll 1
        for (int q = lane; q < nd * nx; q += TG_NL) { const int r = q / nx, i = q - r * nx; W.Ad[r * W.n1 + i] = W.A[i * W.lda + meq + r]; }
    }
    TG_SYNC();
    // ---- unconstrained minimiser xq = -J J' g
    #pragma unroll 1
    for (int k = lane; k < nq; k += TG_NL) {
        double h = 0;
        TG_UNROLL_INNER
        for (int i = 0; i < nq; i++) h += W.Jq[k * ld + i] * (ELIM ? W.rq[i] : W.g[i]);
        W.dq[k] = h;
    }
    TG_SYNC();
    #pragma unroll 1
    for (int i = lane; i < nq; i += TG_NL) {
        double h = 0;
        TG_UNROLL_INNER
        for (int k = 0; k < nq; k++) h += W.Jq[k * ld + i] * W.dq[k];
        if (ELIM) W.sq[i] = -h; else W.xq[i] = -h;
    }
    TG_SYNC();
    // ELIM: lane's entries of the step in the order of x (lane, lane + TG_NL, ...): rotated triple they belong to
    if (ELIM) {
        const double es = -(1 - (coupled ? W.sq[W.nf] : 0.0));
        #pragma unroll 1
        for (int i = lane; i < W.n; i += TG_NL) W.xq[i] = tg_qp_x_entry(W, W.sq, es, i, tg_rot_base(W, i));
        if (nq > n && lane == 0) W.xq[W.n] = W.sq[W.nf];
        TG_SYNC();
    }
    int iq = 0;
    double d2n, dn;
    fl += (double)n * n * n / 3 + 4.0 * nq * nq;          // J = L^-T D^-1/2 ; xq = -J J'g
    // ---- the equality rows in order (outer steps 0 .. meq-1), then the most violated inequality row or bound
    const int itmax = 10 * (nc + nq) + 100;
    #pragma unroll 1
    for (int it = 0; it < itmax + meq; it++) {
        const bool eq = it < meq;
        int ip = it;
        if (ELIM && eq && tg_is_pin_row(W, it)) continue;
        if (!eq) {
            double best = 0;
            ip = 0x7fffffff;
            if (W.nsfc) {
                // corridor rows (lb <= R' Q <= ub, CF/sfc_constraints.py:53-77) through the hull points: lane item =
                // (interval j, hull point k); Q = MINVO point of the step's control points, then the d rotated
                // coordinates serve the d lower and d upper rows of that point -- 4 d + d^2 products for 2 d rows
                // instead of 2 d row products of 4 d terms read from A.  (The row that is picked is re-evaluated from
                // A by tg_qp_value; the scan only ranks violations.)
                const int npts = W.sfc_npts, D = W.cpd, N = W.cpN;
                const double slack = nq > n ? W.xq[W.n] : 0.0;
                #pragma unroll 1
                for (int q = lane; q < npts; q += TG_NL) {
                    const int j = q >> 2, k = q & 3;
                    const double m0 = tg_minvo_py_t(0, k), m1 = tg_minvo_py_t(1, k), m2 = tg_minvo_py_t(2, k), m3 = tg_minvo_py_t(3, k);
                    double Q[3], Qa[3];
                    #pragma unroll
                    for (int c = 0; c < 3; c++) {
                        Q[c] = 0; Qa[c] = 0;
                        if (c < D) {
                            const double *xp = W.xq + c * N + j;
                            const double t0 = xp[0] * m0, t1 = xp[1] * m1, t2 = xp[2] * m2, t3 = xp[3] * m3;
                            Q[c] = t0 + t1 + t2 + t3;
                            Qa[c] = fabs(t0) + fabs(t1) + fabs(t2) + fabs(t3);
                        }
                    }
                    const double *rot = W.rotq + j * D * D;
                    // (the right-hand sides of this point's 2 d rows up front: they come from the persistent state,
                    // which sits in global memory when the kernel does not stage it)
                    double cpv[6];
                    #pragma unroll
                    for (int rr = 0; rr < 3; rr++)
                        #pragma unroll
                        for (int side = 0; side < 2; side++)
                            cpv[2 * rr + side] = rr < D ? W.c[W.sfc0 + side * W.nsfc + rr * npts + q] : 0.0;
                    #pragma unroll
                    for (int rr = 0; rr < 3; rr++) {
                        if (rr >= D) continue;
                        double sq = 0, sa = 0;
                        #pragma unroll
                        for (int c = 0; c < 3; c++)
                            if (c < D) { const double rc = rot[rr * D + c]; sq += rc * Q[c]; sa += fabs(rc) * Qa[c]; }
                        #pragma unroll
                        for (int side = 0; side < 2; side++) {
                            const int p = W.sfc0 + side * W.nsfc + rr * npts + q;
                            if (W.iact[p]) continue;
                            const double cp = cpv[2 * rr + side];
                            double h = side ? -sq : sq, sc = fabs(cp) + sa;
                            if (nq > n) { const double t = fmax(-cp, 0.0) * slack; h += t; sc += fabs(t); }
                            const double sv = h + cp;
                            if (sv < -1e-13 * sc && (sv < best || (sv == best && p < ip))) { best = sv; ip = p; }
                        }
                    }
                }
            }
            // the other rows and the bounds, handed out from the last lane down: the dense rows come first and land on
            // the lanes (of a 64-lane group: on the warp) that the hull points above leave idle
            const int nskip = 2 * W.nsfc;
            #pragma unroll 1
            for (int t = meq + (TG_NL - 1 - lane); t < nc - nskip; t += TG_NL) {
                const int p = t >= W.sfc0 ? t + nskip : t;
                if (W.iact[p]) continue;
                double sv, tol;
                if (p < m) {
                    const int pa = t;          // row of A: the corridor rows are not stored
                    double h = 0, sc = fabs(W.c[p]);
                    if (ELIM && nd > 0 && nd <= 4) {
                        const double *ar = W.Ad + (pa - meq) * W.n1;
                        TG_PRAGMA(unroll TG_DENSE_UNROLL)
                        for (int i = 0; i < nx; i++) { const double t = ar[i] * W.xq[i]; h += t; sc += fabs(t); }
                    } else {
                        TG_PRAGMA(unroll TG_DENSE_FAR_UNROLL)
                        for (int i = 0; i < nx; i++) { const double t = W.A[i * W.lda + pa] * W.xq[i]; h += t; sc += fabs(t); }
                    }
                    sv = h + W.c[p];
                    tol = 1e-13 * sc;
                } else {
                    const int q = p - m;
                    const int i = q < W.n1 ? q : q - W.n1;
                    if (i >= nx) continue;
                    const double bnd = q < W.n1 ? W.u[i] : W.v[i];
                    if (!tg_finite(bnd)) continue;
                    sv = q < W.n1 ? W.xq[i] - bnd : bnd - W.xq[i];
                    tol = 1e-13 * (fabs(bnd) + fabs(W.xq[i]));
                }
                if (sv < -tol && (sv < best || (sv == best && p < ip))) { best = sv; ip = p; }
            }
            tg_wargmin(best, ip);
            fl += 3.0 * ((m - meq - 2 * W.nsfc) * nq + W.sfc_npts * (4 * W.cpd + W.cpd * W.cpd)) + 4.0 * W.nsfc;
            if (ip == 0x7fffffff) {
                #pragma unroll 1
                for (int k = lane; k < iq; k += TG_NL) W.r[W.act[k]] = W.uq[k];
                // rows with a (possibly) non-zero multiplier, for the A'r products of the outer iteration
                int cnt = 0;
                #pragma unroll 1
                for (int k = 0; k < iq; k++)
                    if (W.act[k] < m) { if (lane == 0) W.ract[cnt] = W.act[k]; cnt++; }
                nract = cnt;
                TG_SYNC();
                if (ELIM && pins) {
                    // multipliers of the pin rows, from the pinned variables' entries of B d + g = sum of normals x multipliers
                    // (B d over all variables, QP order; W.Lm: the solve has overwritten the copy of L next to J)
                    #pragma unroll 1
                    const double ys = coupled ? W.sq[W.nf] : 0.0;
                    #pragma unroll 1
                    for (int k = lane; k < W.n; k += TG_NL) {
                        W.hw[k] = k < W.nf ? W.sq[k] : -(1 - ys) * W.w[k - W.nf];
                        if (ident) W.dq[k] = W.hw[k];
                    }
                    TG_SYNC();
                    if (!ident) tg_ldl_apply_tail(W.n, W.Lm, W.Dd, W.hw, W.z, W.dq, W.n, W.nf);
                    #pragma unroll 1
                    for (int e = lane; e < W.ne; e += TG_NL) {
                        const int i = W.perm[W.nf + e];
                        double h = W.dq[W.nf + e] + tg_rot_get(W, W.g, i);
                        #pragma unroll 1
                        for (int k = 0; k < iq; k++)
                            if (W.act[k] < m) h -= tg_normal_entry_r(W, meq, W.act[k], i) * W.uq[k];
                        W.r[tg_pin_row(W, e)] = h / tg_pin_sigma(W, e);
                    }
                    TG_SYNC();
                }
                return TG_QP_OK;
            }
        }
        tg_qp_normal<ELIM>(W, nq, meq, ip, W.np, coupled);
        double uip = 0;
        double sv = tg_qp_value<ELIM>(W, nq, meq, ip, pins);
        #pragma unroll 1
        for (int inner = 0; inner < itmax; inner++) {
            tg_qp_directions(W, nq, iq, d2n, dn);
            fl += 2.0 * nq * nq + 2.0 * nq * (nq - iq) + (double)iq * iq + 4.0 * nq;
            // dual step length: active inequalities whose multiplier would turn negative
            double t1 = INFINITY; int l = 0x7fffffff;
            if (!eq) {
                #pragma unroll 1
                for (int k = lane; k < iq; k += TG_NL)
                    if (W.act[k] >= meq && W.rq[k] > 0) {
                        const double t = W.uq[k] / W.rq[k];
                        if (t < t1) { t1 = t; l = k; }
                    }
                tg_wargmin(t1, l);
            }
            const bool indep = d2n > EPS_DEP * dn;
            if (eq && !indep) return 6;
            const double t2 = indep ? -sv / d2n : INFINITY;
            const double t = t1 < t2 ? t1 : t2;
            if (!(t < INFINITY)) return 4;
            #pragma unroll 1
            for (int k = lane; k < iq; k += TG_NL) W.uq[k] -= t * W.rq[k];
            uip += t;
            const bool primal = t2 < INFINITY;
            if (primal)
                #pragma unroll 1
                for (int i = lane; i < nq; i += TG_NL) { if (ELIM) W.sq[i] += t * W.z[i]; else W.xq[i] += t * W.z[i]; }
#ifdef TG_XQ_INCREMENTAL
            if (ELIM && primal) {
                // the same step in the order of x (eliminated coordinates move with the slack in the coupled problem)
                const double es = coupled ? W.z[n] : 0.0;
                #pragma unroll 1
                for (int i = lane; i < W.n; i += TG_NL) W.xq[i] += t * tg_qp_x_entry(W, W.z, es, i, tg_rot_base(W, i));
                if (nq > n && lane == 0) W.xq[W.n] += t * W.z[n];
            }
            TG_SYNC();
#else
            TG_SYNC();
            if (ELIM && primal) {
                // the point in the order of x, for the scans (formed from the point itself, not step by step: the scans and
                // tg_qp_value must see the same point to the last bits)
                const double es = -(1 - (coupled ? W.sq[W.nf] : 0.0));
                #pragma unroll 1
                for (int i = lane; i < W.n; i += TG_NL) W.xq[i] = tg_qp_x_entry(W, W.sq, es, i, tg_rot_base(W, i));
                if (nq > n && lane == 0) W.xq[W.n] = W.sq[W.nf];
                TG_SYNC();
            }
#endif
            if (primal && t2 <= t1) {
                if (lane == 0) { W.uq[iq] = uip; W.act[iq] = ip; W.iact[ip] = 1; }
                TG_SYNC();
                tg_qp_add(W, nq, iq, d2n);
                fl += 2.0 * nq * (nq - iq) + 3.0 * nq;
                iq++;
                break;
            }
            fl += 6.0 * (iq - 1 - l) * (nq + 0.5 * (iq - 1 - l));
            tg_qp_drop(W, nq, iq, l);
            if (primal) {
                sv = tg_qp_value<ELIM>(W, nq, meq, ip, pins);
                if (inner == itmax - 1) return 3;
            }
        }
    }
    return 3;
}

// sum of constraint violations / L1 penalty term
TG_HD double tg_violation(const TgSqpWs &W, int meq, const double *weights)
{
    double h = 0;
    TG_PRAGMA(unroll TG_VIOL_UNROLL)
    for (int j = TG_LANE(); j < W.m; j += TG_NL) {
        const double cj = W.c[j];
        const double viol = j < meq ? fmax(-cj, cj) : fmax(-cj, 0.0);
        h += weights ? weights[j] * viol : viol;
    }
    return tg_wsum(h);
}

#define TG_SQP_FD_JACOBIAN 1     // flags bit 0: finite-difference emulation instead of analytic derivatives

// objective and constraints at W.x; with derivs also g and the nonlinear rows of A (analytic)
template <int D>
TG_FN double tg_sqp_evaluate(const TgLayout &L, const int *sp, const double *par, const TgSqpWs &W, bool derivs)
{
    const double f = tg_objective(L, sp, W.x, derivs ? W.g : 0);
    TgJac sink = {W.A, 1, W.lda, 2};
    tg_constraints_d<D>(L, sp, par, W.x, W.c, derivs ? &sink : 0, W.scratch);
    TG_SYNC();
    return f;
}

// Derivatives exactly as the reference obtains them: scipy's approx_derivative('2-point',
// abs_step=eps, bounds) on the objective and on every nonlinear constraint
// (scipy/optimize/_slsqp_py.py:353-366, _numdiff.py); linear rows keep their constant A.
// Requires f, W.c at W.x.  n extra evaluations.
template <int D>
TG_FN void tg_sqp_fd_derivatives(const TgLayout &L, const int *sp, const double *par, const TgSqpWs &W, double f)
{
    const int lane = TG_LANE(), n = L.n, m = L.m;
    // the objective and the light blocks: one perturbed evaluation per variable
    #pragma unroll 1
    for (int i = 0; i < n; i++) {
        // a pinned control point that has reached its value does not move any more and its column of the derivatives is
        // not used any more (tg_sqp_stage_qp: its block of B is frozen): no evaluation for it
        if (W.ne && W.ctl->pins_hold && i < W.cpd * W.cpN) {
            const int j = i % W.cpN;
            if ((W.esk && j < 3) || (W.eek && j >= W.cpN - 3)) continue;
        }
        const double xi = W.x[i];
        const double h = tg_fd_step(xi, W.xl[i], W.xu[i]);
        TG_SYNC();
        if (lane == 0) W.x[i] = xi + h;
        TG_SYNC();
        const double dx = W.x[i] - xi;
        const double f1 = tg_objective(L, sp, W.x, 0);
        tg_constraints_d<D>(L, sp, par, W.x, W.cf, 0, W.scratch, TG_SKIP_LINEAR | TG_SKIP_TURNING | TG_SKIP_OBSTACLES);
        TG_SYNC();
        if (lane == 0) { W.g[i] = (f1 - f) / dx; W.x[i] = xi; }
        #pragma unroll 1
        for (int j = L.r_sder + lane; j < L.r_turn; j += TG_NL) W.A[i * W.lda + j] = (W.cf[j] - W.c[j]) / dx;
        TG_SYNC();
    }
    // the heavy blocks: item-parallel sweeps (tg_eval.h)
    if (L.n_turn) tg_fd_turning<D>(L, sp, par, W.x, W.xl, W.xu, W.c[L.r_turn], W.A, W.lda, W.scratch);
    if (L.n_obs) tg_fd_obstacles<D>(L, par, W.x, W.xl, W.xu, W.c, W.A, W.lda, L.r_obs - 2 * L.n_sfc, W.scratch);
    (void)m;
}

// ---------------------------------------------------------------------------
// The iteration, split into two stages so that it can run either fused (one warp loops over both stages
// until its problem is done) or in lock step (all problems run stage LS, then all run stage QP, ... as
// separate kernels: every warp of the machine then executes the same, small piece of code at the same time).
//   stage LS : evaluation at the starting point / the whole line search on the L1 merit function
//   stage QP : convergence test after the step, damped BFGS update, next QP subproblem, merit set-up
// ---------------------------------------------------------------------------
TG_FN void tg_sqp_begin(const TgLayout &L, const TgSqpWs &W, const double *xin, int maxiter, double acc, int flags)
{
    const int lane = TG_LANE(), n = L.n, m = L.m, n1 = W.n1;
    // variables and bounds (TG/objectives/objective_variables.py:50-61); x0 clipped as scipy does
    #pragma unroll 1
    for (int i = lane; i < n1; i += TG_NL) {
        double lo = -INFINITY, hi = INFINITY;
        if (i >= L.ia && i < L.it0) lo = 10e-8;
        if (i >= L.it0 && i < n) { lo = 0; hi = L.N - 3; }
        W.xl[i] = lo; W.xu[i] = hi;
        double xv = i < n ? xin[i] : 0.0;
        if (i < n) { xv = xv < lo ? lo : xv; xv = xv > hi ? hi : xv; }
        W.x[i] = xv; W.s[i] = 0; W.g[i] = 0; W.x0[i] = xv; W.gl[i] = 0;
    }
    #pragma unroll 1
    for (int j = lane; j < m; j += TG_NL) W.mu[j] = 0;
    #pragma unroll 1
    for (int q = lane; q < W.lda * n1; q += TG_NL) W.A[q] = 0;
    if (lane == 0) {
        TgSqpCtl c;
        c.f = 0; c.f0 = 0; c.t0 = 0; c.h3 = 0; c.h4 = 1; c.alpha = 1; c.acc = acc; c.flops = 0;
        c.state = TG_ST_INIT; c.iter = 0; c.ireset = 0; c.line = 0; c.badlin = 0; c.nfev = 0; c.status = -1;
        c.need_reset = 1; c.maxiter = maxiter; c.flags = flags; c.nract = 0; c.need_der = 0; c.pins_hold = 0;
        *W.ctl = c;
    }
    TG_SYNC();
}

// The stage is written against an evaluator `ev` -- ev.init(W): constant rows of A and whatever the QP stage needs
// once; ev.value(W): objective at W.x (return value) and constraint rows into W.c -- so that other problem kinds
// (the spline order converter, tg_smooth.cu) run the same line search; the trajectory evaluator is TgTrajectoryEval.
template <class Ev>
TG_HD void tg_sqp_stage_ls_t(const TgLayout &L, const TgSqpWs &W, const Ev &ev, double *trace, int trace_cap)
{
    const int lane = TG_LANE(), n = L.n, meq = L.meq;
    TgSqpCtl ctl = *W.ctl;
    const bool init = ctl.state == TG_ST_INIT;
    if (init || ctl.state == TG_ST_LS) {
        if (init) ev.init(W);
        // one evaluation at the starting point, or the whole line search on the L1 merit function
        double f;
        #pragma unroll 1
        for (;;) {
            f = ev.value(W);
            ctl.nfev++;
            if (init) break;
            const double t = f + tg_violation(W, meq, W.mu);
            const double h1 = t - ctl.t0;
            if (h1 <= ctl.h3 / 10 || ctl.line > 10) break;
            ctl.alpha = fmax(ctl.h3 / (2 * (ctl.h3 - h1)), 0.1);
            ctl.line++;
            ctl.h3 = ctl.alpha * ctl.h3;
            TG_SYNC();
            #pragma unroll 1
            for (int i = lane; i < n; i += TG_NL) {
                W.s[i] *= ctl.alpha;
                double xv = W.x0[i] + W.s[i];
                xv = xv < W.xl[i] ? W.xl[i] : xv;
                xv = xv > W.xu[i] ? W.xu[i] : xv;
                W.x[i] = xv;
            }
            TG_SYNC();
        }
        ctl.f = f;
        if (!init && trace && lane == 0 && (ctl.iter * (n + 2) <= trace_cap)) {
            double *tr = trace + (ctl.iter - 1) * (n + 2);
            tr[0] = f; tr[1] = ctl.alpha;
            for (int i = 0; i < n; i++) tr[2 + i] = W.x[i];
        }
        // scipy differentiates at the accepted point only (mode -1) -> stage DER; harmless extra work if the next
        // test ends the run
        ctl.need_der = 1;
        ctl.state = init ? TG_ST_QP : TG_ST_UPDATE;
    }
    TG_SYNC();
    if (lane == 0) *W.ctl = ctl;
    TG_SYNC();
}

template <int D>
struct TgTrajectoryEval {
    const TgLayout &L;
    const int *sp;
    const double *par;
    TG_MEMBER void init(const TgSqpWs &W) const
    {
        TgJac sink = {W.A, 1, W.lda, 2};
        tg_linear_jacobian_d<D>(L, sp, par, sink);
        // rotation of the corridor that owns each interval, for the QP stage's violation scans
        if (L.n_sfc) {
            #pragma unroll 1
            for (int q = TG_LANE(); q < L.nint * D * D; q += TG_NL) {
                const int j = q / (D * D);
                W.rot[q] = par[L.p_sfc + tg_corridor_of_interval(sp, j) * tg_sfc_stride(D) + (q - j * D * D)];
            }
        }
    }
    TG_MEMBER double value(const TgSqpWs &W) const { return tg_sqp_evaluate<D>(L, sp, par, W, false); }
};

template <int D>
TG_FN void tg_sqp_stage_ls(const TgLayout &L, const int *sp, const double *par, const TgSqpWs &W, double *trace,
                           int trace_cap)
{
    const TgTrajectoryEval<D> ev = {L, sp, par};
    tg_sqp_stage_ls_t(L, W, ev, trace, trace_cap);
}

// stage DER: derivatives at the point stage LS accepted -- the analytic gradient and Jacobian rows (values are
// recomputed on the way: same numbers), or scipy's forward differences in finite-difference mode
template <int D>
TG_FN void tg_sqp_stage_der(const TgLayout &L, const int *sp, const double *par, const TgSqpWs &W)
{
    TgSqpCtl ctl = *W.ctl;
    if (!ctl.need_der) return;
    if (ctl.flags & TG_SQP_FD_JACOBIAN) {
        tg_sqp_fd_derivatives<D>(L, sp, par, W, ctl.f);
        ctl.nfev += L.n;
    } else {
        const double f = tg_objective(L, sp, W.x, W.g);
        TgJac sink = {W.A, 1, W.lda, 2};
        tg_constraints_d<D>(L, sp, par, W.x, W.c, &sink, W.scratch);
        TG_SYNC();
        (void)f;
    }
    ctl.need_der = 0;
    TG_SYNC();
    if (TG_LANE() == 0) *W.ctl = ctl;
    TG_SYNC();
}

// copy of the factor between its home and J's storage; `wide`: 16-byte accesses where both ends allow them
TG_HD void tg_copy_doubles(double *dst, const double *src, int count, bool wide)
{
    const int lane = TG_LANE();
#ifdef __CUDA_ARCH__
    if (wide && ((((size_t)dst) | ((size_t)src)) & 15) == 0) {
        double2 *d2 = reinterpret_cast<double2 *>(dst);
        const double2 *s2 = reinterpret_cast<const double2 *>(src);
        #pragma unroll 2
        for (int q = lane; q < count / 2; q += TG_NL) d2[q] = s2[q];
        if ((count & 1) && lane == 0) dst[count - 1] = src[count - 1];
        return;
    }
#endif
    (void)wide;
    #pragma unroll 4
    for (int q = lane; q < count; q += TG_NL) dst[q] = src[q];
}

// lm_far: the persistent state (W.Lm ...) lives in global memory (lock-step kernel of a shape whose state is not
// staged in shared memory).  The factor L is then copied once into the storage of J (free until the QP is set up),
// updated there, written back once and handed to the QP set-up from there, instead of being read five times and
// written twice through L2.  Same arithmetic.
// SPLIT_NQ (instantiations with a compile-time descriptor): the plain subproblem (n variables) and the augmented one
// (n + 1) get a copy of the solver each, so that the plain one -- all but a few per cent of the calls -- runs with a
// constant number of variables: loop bounds of the products known, no remainder handling.
template <bool LM_FAR, bool SPLIT_NQ = false>
TG_QFN void tg_sqp_stage_qp(const TgLayout &L, const TgSqpWs &W)
{
    // the update's scratch (5 n doubles) comes from R's storage when L sits in J's
    const bool lm_far = LM_FAR && (W.ne || W.n1 * (W.n1 + 1) / 2 + 1 >= 5 * L.n);
    const bool elim = W.ne > 0;          // pinned variables: the factor of B and the update's vectors are in QP order
    bool lcopy = false;      // J's storage holds the current L
    bool ident = false;      // the factor has been reset in this call: B = I
    const int lane = TG_LANE(), n = L.n, m = L.m, meq = L.meq, n1 = W.n1;
    TgSqpCtl ctl = *W.ctl;
    const double acc = ctl.acc, tol = 10 * ctl.acc;
    double h1, h2, h3;
    double fl = 0;       // model count of the stage's fp64 operations (2 per multiply-add), for the roofline report
    if (W.nsfc) {
        // rotation of the corridor that owns each interval: regenerates corridor normals and serves the violation scans
        #pragma unroll 1
        for (int q = lane; q < (W.sfc_npts >> 2) * W.cpd * W.cpd; q += TG_NL) W.rotq[q] = W.rot[q];
        TG_SYNC();
    }
    if (elim) {
        #pragma unroll 1
        for (int i = lane; i < n; i += TG_NL) { const int k = tg_qp_index(W, i); W.perm[k] = i; W.qix[i] = k; }
        TG_SYNC();
    }
    if (ctl.state == TG_ST_UPDATE) {
        // ---- convergence test after the step
        double sn = 0;
        #pragma unroll 1
        for (int i = lane; i < n; i += TG_NL) sn += W.s[i] * W.s[i];
        sn = sqrt(tg_wsum(sn));
        h3 = tg_violation(W, meq, 0);
        if ((fabs(ctl.f - ctl.f0) < acc || sn < acc) && h3 < acc && !ctl.badlin && ctl.f == ctl.f) {
            ctl.status = 0; ctl.state = TG_ST_DONE;
        } else {
            // ---- damped BFGS update of L D L' (derivatives at the new point are already in g, A)
            if (elim) {
                // (active rows and their multipliers first, side by side in the QP's scratch: the loop below then waits
                // on one trip to the persistent state instead of one per active row)
                #pragma unroll 1
                for (int k = lane; k < ctl.nract; k += TG_NL) { const int j = W.ract[k]; W.act[k] = j; W.uq[k] = W.r[j]; }
                TG_SYNC();
            }
            #pragma unroll 1
            for (int i = lane; i < n; i += TG_NL) {
                double h = W.g[i];
                if (elim) {
                    TG_PRAGMA(unroll TG_LAG_UNROLL)
                    for (int k = 0; k < ctl.nract; k++) {
                        const int j = W.act[k];
                        h -= (tg_is_sfc_row(W, j) ? tg_sfc_entry(W, W.rotq, j, i) : W.A[i * W.lda + tg_arow(W, j)]) * W.uq[k];
                    }
                    W.v[i] = h - W.gl[i];           // (order of x; taken to QP order below)
                } else {
                    TG_PRAGMA(unroll TG_LAG_FAR_UNROLL)
                    for (int k = 0; k < ctl.nract; k++) {
                        const int j = W.ract[k];
                        h -= (tg_is_sfc_row(W, j) ? tg_sfc_entry(W, W.rotq, j, i) : W.A[i * W.lda + tg_arow(W, j)]) * W.r[j];
                    }
                    W.u[i] = h - W.gl[i];
                }
            }
            const double *sq = elim ? W.sq : W.s;         // the step in the order of the factor
            TG_SYNC();
            if (elim) {
                #pragma unroll 1
                for (int i = lane; i < n; i += TG_NL) {
                    const int k = tg_qp_index(W, i);
                    W.u[k] = tg_rot_get(W, W.v, i); W.sq[k] = tg_rot_get(W, W.s, i);
                }
                TG_SYNC();
            }
            // Once the eliminated coordinates have reached their values their steps are zero for good, and their rows
            // and columns of B never enter a subproblem again: only the leading nf x nf block of the factor (QP order)
            // is updated from then on -- the same free block in exact arithmetic.
            const int nb = (elim && ctl.pins_hold) ? W.nf : n;
            if (lm_far) {
                tg_copy_doubles(W.Jq, W.Lm, nb * n, elim);
                TG_SYNC();
                lcopy = true;
                tg_ldl_apply(nb, W.Jq, W.Dd, sq, W.w, W.v, n);
            } else tg_ldl_apply(nb, W.Lm, W.Dd, sq, W.w, W.v, n);
            h1 = 0; h2 = 0;
            #pragma unroll 1
            for (int i = lane; i < nb; i += TG_NL) { h1 += sq[i] * W.u[i]; h2 += sq[i] * W.v[i]; }
            tg_wsum2(h1, h2);
            h3 = 0.2 * h2;
            if (h1 < h3) {
                const double h4 = (h2 - h3) / (h2 - h1);
                h1 = h3;
                #pragma unroll 1
                for (int i = lane; i < nb; i += TG_NL) W.u[i] = h4 * W.u[i] + (1 - h4) * W.v[i];
            }
            TG_SYNC();
            fl += 2.0 * n * ctl.nract + 6.0 * n * n + 8.0 * n;         // u = grad L - gl ; v = B s ; two rank-one updates of L D L'
            if (h1 == 0 || h2 == 0) ctl.need_reset = 1;
            else {
                #pragma unroll 1
                // (scratch of the update: 5 n doubles; with L in J's storage they come from R's, free until the QP set-up)
                for (int pass = 0; pass < 2; pass++) {
                    if (lm_far) tg_ldl_update(nb, pass == 0 ? 1 / h1 : -1 / h2, pass == 0 ? W.u : W.v, W.Jq, W.Dd, W.w, W.usc, n);
                    else tg_ldl_update(nb, pass == 0 ? 1 / h1 : -1 / h2, pass == 0 ? W.u : W.v, W.Lm, W.Dd, W.w, elim ? W.usc : W.Jq, n);
                }
                if (lm_far) {
                    tg_copy_doubles(W.Lm, W.Jq, nb * n, elim);
                    TG_SYNC();
                }
                if (elim && W.nsfc) {
                    // (the update's scratch reached into the rotation table)
                    #pragma unroll 1
                    for (int q = lane; q < (W.sfc_npts >> 2) * W.cpd * W.cpd; q += TG_NL) W.rotq[q] = W.rot[q];
                    TG_SYNC();
                }
            }
            ctl.state = TG_ST_QP;
        }
    }
    if (ctl.state == TG_ST_QP) {
        do {
            if (ctl.need_reset) {
                // ---- reset the BFGS factor to the identity
                ctl.ireset++;
                if (ctl.ireset > 5) {
                    // relaxed convergence test after a positive directional derivative
                    double sn = 0;
                    #pragma unroll 1
                    for (int i = lane; i < n; i += TG_NL) sn += W.s[i] * W.s[i];
                    sn = sqrt(tg_wsum(sn));
                    h3 = tg_violation(W, meq, 0);
                    ctl.status = ((fabs(ctl.f - ctl.f0) < tol || sn < tol) && h3 < tol && !ctl.badlin && ctl.f == ctl.f) ? 0 : 8;
                    ctl.state = TG_ST_DONE;
                    break;
                }
                #pragma unroll 1
                lcopy = false;
                for (int q = lane; q < n * n; q += TG_NL) W.Lm[q] = 0;
                #pragma unroll 1
                for (int i = lane; i < n1; i += TG_NL) W.Dd[i] = 1;
                TG_SYNC();
                ctl.need_reset = 0;
                ident = true;
            }
            // ---- major iteration
            ctl.iter++;
            if (ctl.iter > ctl.maxiter) { ctl.status = 9; ctl.state = TG_ST_DONE; break; }
            #pragma unroll 1
            for (int i = lane; i < n; i += TG_NL) { W.u[i] = W.xl[i] - W.x[i]; W.v[i] = W.xu[i] - W.x[i]; }
            TG_SYNC();
            ctl.h4 = 1;
            ctl.badlin = 0;
            // attempt 0: the QP itself.  Attempts 1-6 (SLSQP): if its linearised constraints are inconsistent, the
            // augmented problem with one slack variable, penalty 100, x10 per retry.  Attempt 7 (last resort, departs
            // from SLSQP, which exits here): the dual active-set method works on the inverse factor L^-T D^-1/2 and
            // loses the subproblem when D spans ~20 orders of magnitude, where scipy's least-squares chain carries
            // on; one more try on the augmented problem with D floored at 1e-10 of its largest entry keeps such
            // problems iterating the way the reference does.
            int mode = 0, nq = n;
            double rho = 0, dfloor = 0;
            bool moving = false;
            #pragma unroll 1
            for (int attempt = 0; attempt < 8; attempt++) {
                if (attempt >= 1 && nq == n) {
                    ctl.badlin = 1;
                    #pragma unroll 1
                    for (int j = lane; j < m; j += TG_NL)
                        if (!tg_is_sfc_row(W, j)) W.A[n * W.lda + tg_arow(W, j)] = tg_slack_coeff(W, meq, j);
                    if (lane == 0) { W.g[n] = 0; W.u[n] = 0; W.v[n] = 1; }
                    TG_SYNC();
                    nq = n1;
                }
                if (attempt >= 1) rho = attempt == 1 || attempt == 7 ? 100 : rho * 10;
                if (attempt == 7) {
                    double dmax = 0;
                    #pragma unroll 1
                    for (int i = 0; i < n; i++) dmax = fmax(dmax, W.Dd[i]);
                    dfloor = 1e-10 * dmax;
                }
                // (one call site per number of variables: the solver is inlined.  Only its first loop, which packs L next
                // to J, reads Lsrc)
                const double *Lsrc = (lm_far && lcopy) ? W.Jq : W.Lm;
                if (elim) {
                    if (SPLIT_NQ && nq == n) mode = tg_qp_solve<true>(W, Lsrc, W.nf, meq, rho, fl, ctl.nract, dfloor, ident, ctl.pins_hold != 0, moving);
                    else mode = tg_qp_solve<true>(W, Lsrc, nq == n ? W.nf : W.nf + 1, meq, rho, fl, ctl.nract, dfloor, ident, ctl.pins_hold != 0, moving);
                } else if (SPLIT_NQ && nq == n) mode = tg_qp_solve<false>(W, Lsrc, n, meq, rho, fl, ctl.nract, dfloor, ident, ctl.pins_hold != 0, moving);
                else mode = tg_qp_solve<false>(W, Lsrc, nq, meq, rho, fl, ctl.nract, dfloor, ident, ctl.pins_hold != 0, moving);
                lcopy = false;        // the copy shared J's storage: the solve has overwritten it
                if (attempt == 0 && mode == 6 && n == meq) mode = 4;
                if (mode == TG_QP_OK) break;
                if (mode != 4 && attempt < 6) attempt = 6;          // exits 6 / 3: straight to the last resort
            }
#if defined(TG_QP_DEBUG) && !defined(__CUDA_ARCH__)
            {
                double dmin = 1e300, dmax = 0;
                for (int i = 0; i < n; i++) { dmin = fmin(dmin, W.Dd[i]); dmax = fmax(dmax, W.Dd[i]); }
                printf("iter %3d mode %d badlin %d rho %.0e  D in [%.2e, %.2e]  f %.8g hold %d moving %d\n", ctl.iter, mode, ctl.badlin, rho, dmin, dmax, ctl.f, ctl.pins_hold, (int)moving);
            }
#endif
            if (mode != TG_QP_OK) { ctl.status = mode; ctl.state = TG_ST_DONE; break; }
            // (shapes with pinned control points only: with rotated triples alone the saving is a few per cent of the
            // factor update, and nothing in the derivative stage)
            if (elim && (W.esk | W.eek) && !moving) ctl.pins_hold = 1;
            if (ctl.badlin) ctl.h4 = 1 - W.xq[n];
            // ---- gradient of the Lagrangian at the old point, merit weights
            if (elim) {
                #pragma unroll 1
                for (int k = lane; k < ctl.nract; k += TG_NL) { const int j = W.ract[k]; W.act[k] = j; W.uq[k] = W.r[j]; }
                TG_SYNC();
            }
            #pragma unroll 1
            for (int i = lane; i < n; i += TG_NL) {
                double h = W.g[i];
                if (elim) {
                    TG_PRAGMA(unroll TG_LAG_UNROLL)
                    for (int k = 0; k < ctl.nract; k++) {
                        const int j = W.act[k];
                        h -= (tg_is_sfc_row(W, j) ? tg_sfc_entry(W, W.rotq, j, i) : W.A[i * W.lda + tg_arow(W, j)]) * W.uq[k];
                    }
                } else {
                    TG_PRAGMA(unroll TG_LAG_FAR_UNROLL)
                    for (int k = 0; k < ctl.nract; k++) {
                        const int j = W.ract[k];
                        h -= (tg_is_sfc_row(W, j) ? tg_sfc_entry(W, W.rotq, j, i) : W.A[i * W.lda + tg_arow(W, j)]) * W.r[j];
                    }
                }
                W.gl[i] = h;
                W.s[i] = W.xq[i];
                W.x0[i] = W.x[i];
            }
            ctl.f0 = ctl.f;
            fl += 2.0 * n * ctl.nract + 8.0 * m + 4.0 * n;
            TG_SYNC();
            double gs = 0;
            #pragma unroll 1
            for (int i = lane; i < n; i += TG_NL) gs += W.g[i] * W.s[i];
            gs = tg_wsum(gs);
            h1 = 0; h2 = 0;
            TG_PRAGMA(unroll TG_VIOL_UNROLL)
            for (int j = lane; j < m; j += TG_NL) {
                const double cj = W.c[j];
                h2 += fmax(-cj, j < meq ? cj : 0.0);
                const double ar = fabs(W.r[j]);
                W.mu[j] = fmax(ar, (W.mu[j] + ar) / 2);
                h1 += ar * fabs(cj);
            }
            h1 = fabs(gs) + tg_wsum(h1);
            h2 = tg_wsum(h2);
            TG_SYNC();
            if (h1 < acc && h2 < acc && !ctl.badlin && ctl.f == ctl.f) { ctl.status = 0; ctl.state = TG_ST_DONE; break; }
            h1 = tg_violation(W, meq, W.mu);
            ctl.t0 = ctl.f + h1;
            h3 = gs - h1 * ctl.h4;
            if (h3 >= 0) { ctl.need_reset = 1; break; }       // stays in state QP: the reset costs a major iteration
            // ---- first trial point of the line search (alpha = 1)
            ctl.alpha = 1; ctl.line = 1; ctl.h3 = h3;
            #pragma unroll 1
            for (int i = lane; i < n; i += TG_NL) {
                double xv = W.x0[i] + W.s[i];
                xv = xv < W.xl[i] ? W.xl[i] : xv;
                xv = xv > W.xu[i] ? W.xu[i] : xv;
                W.x[i] = xv;
            }
            ctl.state = TG_ST_LS;
        } while (0);
    }
    ctl.flops += fl;
    TG_SYNC();
    if (lane == 0) *W.ctl = ctl;
    TG_SYNC();
}

// fused driver: one warp runs both stages until its problem is done (host tests; small batches)
template <int D>
TG_FN void tg_sqp_solve(const TgLayout &L, const int *sp, const double *par, double *xio, double *wsbase, int maxiter,
                        double acc, int flags, TgSqpResult *res, double *trace, int trace_cap)
{
    TgSqpWs W;
    tg_sqp_carve(L, wsbase, &W);
    tg_sqp_begin(L, W, xio, maxiter, acc, flags);
    #pragma unroll 1
    for (;;) {
        const int st = W.ctl->state;
        if (st == TG_ST_DONE) break;
        if (st == TG_ST_INIT || st == TG_ST_LS) { tg_sqp_stage_ls<D>(L, sp, par, W, trace, trace_cap); tg_sqp_stage_der<D>(L, sp, par, W); }
#ifdef TG_FUSED_LM_FAR          // host tests of the lock-step kernels' variant of the stage (L worked on in J's storage)
        else tg_sqp_stage_qp<true>(L, W);
#else
        else tg_sqp_stage_qp<false>(L, W);
#endif
    }
    #pragma unroll 1
    for (int i = TG_LANE(); i < L.n; i += TG_NL) xio[i] = W.x[i];
    TG_SYNC();
    if (res && TG_LANE() == 0) {
        res->status = W.ctl->status; res->nit = W.ctl->iter > maxiter ? maxiter : W.ctl->iter;
        res->nfev = W.ctl->nfev; res->f = W.ctl->f;
    }
}

// the reference's is_violation: violation flags of the LAST constraint in its list, tolerance 10e-6
// (TG/trajectory_generator.py:252-261, DS/constraint_function_data.py:12,45-48)
TG_HD int tg_last_block_violation(const TgLayout &L, const double *c)
{
    int r0, r1, eq = 0;
    if (L.n_obs) { r0 = L.r_obs; r1 = r0 + L.n_obs; }
    else if (L.n_sfc) { r0 = L.r_sfcl; r1 = r0 + 2 * L.n_sfc; }
    else if (L.n_turn) { r0 = L.r_turn; r1 = r0 + 1; }
    else if (L.n_tan) { r0 = L.r_tanl; r1 = r0 + 2 * L.n_tan; }
    else if (L.n_db) { r0 = L.r_db; r1 = r0 + L.n_db; }
    else if (L.n_iwv) { r0 = L.r_iwv; r1 = r0 + L.n_iwv; eq = 1; }
    else if (L.n_iwl) { r0 = L.r_iwl; r1 = r0 + L.n_iwl; eq = 1; }
    else if (L.n_eder) { r0 = L.r_eder; r1 = r0 + L.n_eder; eq = 1; }
    else if (L.n_sder) { r0 = L.r_sder; r1 = r0 + L.n_sder; eq = 1; }
    else { r0 = L.r_end; r1 = r0 + L.n_end; eq = 1; }
    int bad = 0;
    #pragma unroll 1
    for (int j = r0 + TG_LANE(); j < r1; j += TG_NL) {
        const double v = c[j];
        if (eq ? (fabs(v) > 10e-6) : (v < -10e-6)) bad = 1;
        if (v != v) bad = 1;
    }
    return tg_any(bad);
}

// ---------------------------------------------------------------------------
// Multipliers and first-order optimality certificate of a finished solve (finish kernel, fused kernel, host build).
// lam[m]: the multipliers of the last QP in row order -- scipy's OptimizeResult.multipliers (mult[:meq] equality rows,
// then the inequality rows; no bound multipliers).  The rows the QP eliminates (tg_sqp_pinned) carry a multiplier only
// while their coordinates still move (tg_qp_solve leaves 0 otherwise); theirs is recovered here from the QP's
// stationarity on the eliminated coordinates, with gl (the Lagrangian gradient the QP stage formed with the last QP's
// multipliers), the bound multipliers and the factor L D L' the QP ran with (see below).  Once the pins hold
// (TgSqpCtl::pins_hold) the factor's pinned rows are frozen, B_Pf is not scipy's, and the recovered multipliers deviate
// by what DESIGN.md records.  For status != 0 lam is the last successful QP's values with the same recovery (exit 9:
// the factor may have been updated after that QP; exits 4 / 6: r is zero); they are not checked against an oracle.
// kkt[4], absolute, NaN -> +inf, with the solver's own derivatives (g, A: analytic or finite-difference, whichever the
// solve ran) at the returned x and gradL = g - sum_j lam_j grad c_j over the rows with lam_j != 0:
//   [0] stationarity  max_i |pi_i|, pi_i = min(gradL_i, 0) at x_i == xl_i, max(gradL_i, 0) at x_i == xu_i, else gradL_i
//   [1] infeasibility max |c_j| (equality rows), max(0, -c_j) (inequality rows)
//   [2] dual infeasibility max(0, -lam_j) over the inequality rows
//   [3] complementarity max |lam_j c_j| over the inequality rows
// Either output may be null.  scratch: tg_sqp_kkt_scratch_doubles(L) doubles (none without eliminated rows).  Every sum
// runs in a fixed order: the results do not depend on the lanes per problem.
// ---------------------------------------------------------------------------
TG_HD size_t tg_sqp_kkt_scratch_doubles(const TgLayout &L) { return tg_sqp_pinned(L) ? (size_t)L.n + (L.n & 1) : 0; }

TG_HD double tg_kkt_fold(double acc, double v) { return v != v ? INFINITY : fmax(acc, v); }

TG_FN void tg_sqp_kkt(const TgLayout &L, const TgSqpWs &W, double *lam, double *kkt, double *scratch)
{
    const int lane = TG_LANE(), n = L.n, m = L.m, meq = L.meq;
    // ---- multipliers of the eliminated rows.  The QP's stationarity in QP order, with d_P = 0 (pins that do not move):
    // B_ff d_f = -v_f and sigma lambda_P = (B d)_P + v_P, v = gl - (bound multipliers) in rotated space.  With
    // B = L D L' (free block leading), B_Pf B_ff^-1 = L_Pf L_ff^-1, so sigma lambda_P = v_P - L_Pf L_ff^-1 v_f: one forward
    // substitution with the free block of the factor, run on into the eliminated rows.  (The stored step s cannot stand
    // in for d: the line search has scaled it by the product of its trial steps.)  Once the pins hold, L_Pf is frozen
    // and the term is dropped: sigma lambda_P = v_P agrees better with the full-space subproblem then (DESIGN.md).
    double *v = W.ne ? scratch : nullptr;
    if (W.ne) {
        #pragma unroll 1
        for (int i = lane; i < n; i += TG_NL) v[tg_qp_index(W, i)] = tg_rot_get(W, W.gl, i) - (W.r[m + i] - W.r[m + W.n1 + i]);
        TG_SYNC();
        if (!W.ctl->pins_hold && TG_SERIAL_ACTIVE()) {
            #pragma unroll 1
            for (int j = 0; j < W.nf; j++) {
                const double yj = v[j];
                #pragma unroll 1
                for (int k = j + 1 + lane; k < n; k += TG_SERIAL_LANES) v[k] -= W.Lm[j * n + k] * yj;
                TG_SERIAL_SYNC();
            }
        }
        TG_SYNC();
        #pragma unroll 1
        for (int e = lane; e < W.ne; e += TG_NL) {
            const double rq = W.r[tg_pin_row(W, e)];          // pins that moved in the last QP: the QP formed it
            v[W.nf + e] = rq != 0 ? rq : v[W.nf + e] / tg_pin_sigma(W, e);
        }
        TG_SYNC();
    }
    if (lam) {
        #pragma unroll 1
        for (int j = lane; j < m; j += TG_NL) lam[j] = W.r[j];
        TG_SYNC();
        #pragma unroll 1
        for (int e = lane; e < W.ne; e += TG_NL) lam[tg_pin_row(W, e)] = v[W.nf + e];
        TG_SYNC();
    }
    if (!kkt) return;
    // ---- stationarity: the rows of the last QP's active set (W.ract; the only rows with r != 0) and the eliminated rows
    double st = 0;
    const int nract = W.ctl->nract;
    #pragma unroll 1
    for (int i = lane; i < n; i += TG_NL) {
        double h = W.g[i];
        #pragma unroll 1
        for (int k = 0; k < nract; k++) {
            const int j = W.ract[k];
            const double rj = W.r[j];
            if (rj != 0) h -= (tg_is_sfc_row(W, j) ? tg_sfc_entry(W, W.rot, j, i) : W.A[i * W.lda + tg_arow(W, j)]) * rj;
        }
        #pragma unroll 1
        for (int e = 0; e < W.ne; e++) {
            const double le = v[W.nf + e];
            if (le != 0) h -= W.A[i * W.lda + tg_arow(W, tg_pin_row(W, e))] * le;
        }
        const double pi = W.x[i] == W.xl[i] ? fmin(h, 0.0) : W.x[i] == W.xu[i] ? fmax(h, 0.0) : h;
        st = tg_kkt_fold(st, fabs(pi));
    }
    // ---- the row folds (the eliminated rows are equality rows: lam_j = r_j over the inequality rows)
    double inf = 0, dinf = 0, comp = 0;
    #pragma unroll 1
    for (int j = lane; j < m; j += TG_NL) {
        const double cj = W.c[j];
        if (j < meq) { inf = tg_kkt_fold(inf, fabs(cj)); continue; }
        const double rj = W.r[j];
        inf = tg_kkt_fold(inf, -cj);
        dinf = tg_kkt_fold(dinf, -rj);
        comp = tg_kkt_fold(comp, fabs(rj * cj));
    }
    int k0 = 0;
    tg_wargmax(st, k0); tg_wargmax(inf, k0); tg_wargmax(dinf, k0); tg_wargmax(comp, k0);
    if (lane == 0) { kkt[0] = st; kkt[1] = inf; kkt[2] = dinf; kkt[3] = comp; }
    TG_SYNC();
}


#endif  // TG_SQP_H
